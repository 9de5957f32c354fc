// sm_100a kernels of the gate-evaluation hot path.
//
// What they replace (reference, rust/src/consumers/evaluator.rs):
//   k_level        one wavefront of PlaintextBackend::{add, multiply, add_constant, mul_constant,
//                  and, xor, not} (:908-938) with `assert_zero` (:900-906) fused into the
//                  producing gate, for a whole tile of witnesses at once
//   k_load_inputs  `constant` / `instance` / `witness` (:896-898, 940-946): raw little-endian
//                  values -> Montgomery residues in the wire store
//   k_read_values  what `Evaluator::get` (:750-752) returns: canonical residues of chosen wires
//   k_level_pipe / k_level_tma   the hot forms of k_level: software-pipelined per-thread vector loads / operand rows
//                  through the bulk-copy engine into an mbarrier ring (8-limb fields, tiles of >= 256 lanes)
//   k_levels_coop  every wavefront in one launch, grid or cluster barrier between them (launch-bound programs)
//   k_levels_flow  every wavefront in one launch with NO barrier: dataflow on marker words (one witness, 1- / 2-limb fields)
//   k_bool_*       the same for p = 2, bit-sliced (32 witnesses per word); k_bool_groups expands the loop-structured
//                  call groups of program.h (For over a plain function, evaluator.rs:495-559 + :441-471 + :698-746)
//
// No tensor cores on purpose: nothing on this path is a dense contraction.  The work is HBM-bound
// streaming of wire limbs plus 32-bit integer multiply-add chains (IMAD), see DESIGN.md.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include <cooperative_groups.h>

#include "device_util.cuh"
#include "kernels.cuh"

namespace cg = cooperative_groups;

namespace zkb {

// ---------------------------------------------------------------------------------------------
// constants: canonical residues -> Montgomery form (once per program upload)
// ---------------------------------------------------------------------------------------------
template <int N>
__global__ void k_to_mont(uint32_t* consts, uint32_t n, FieldParams fp) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t a[N], r[N];
#pragma unroll
    for (int k = 0; k < N; k++) a[k] = consts[(size_t)i * N + k];
    fe_mont_mul<N>(r, a, fp.r2, fp.p, fp.n0inv);
#pragma unroll
    for (int k = 0; k < N; k++) consts[(size_t)i * N + k] = r[k];
}

// ---------------------------------------------------------------------------------------------
// inputs: raw LE bytes -> Montgomery residues, witness-minor
// ---------------------------------------------------------------------------------------------
template <int N>
__global__ void __launch_bounds__(256)
k_load_inputs(const InputLoad* __restrict__ loads, uint32_t n_loads, uint32_t* __restrict__ store,
              const uint32_t* __restrict__ consts_mont, InputDesc in, TileGeom g, uint32_t* unreduced_count,
              uint8_t* __restrict__ rawflag, const uint8_t* __restrict__ const_flags, FieldParams fp) {
    const uint64_t total = (uint64_t)n_loads << g.log2_wt;
    const uint32_t wt_mask = (1u << g.log2_wt) - 1;
    for (uint64_t tid = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; tid < total;
         tid += (uint64_t)gridDim.x * blockDim.x) {
        uint32_t lane = (uint32_t)tid & wt_mask;
        InputLoad ld = loads[tid >> g.log2_wt];
        uint32_t v[N];
        bool raw_ge_p = false;  // the reference would hold this input unreduced (raw integer >= p)
#pragma unroll
        for (int k = 0; k < N; k++) v[k] = 0;
        if (lane < g.n_valid) {
            if (ld.kind == V_CONST) {
#pragma unroll
                for (int k = 0; k < N; k++) v[k] = consts_mont[(size_t)ld.index * N + k];
                raw_ge_p = const_flags != nullptr && const_flags[ld.index] != 0;
            } else {
                const uint8_t* src = (ld.kind == V_INSTANCE)
                                         ? in.inst + (uint64_t)(g.batch0 + lane) * in.inst_set_stride
                                         : in.wit + (uint64_t)(g.batch0 + lane) * in.wit_set_stride;
                src += (uint64_t)ld.index * in.stride;
                load_raw_value<N>(v, raw_ge_p, src, in.stride, fp);
                if (raw_ge_p) atomicAdd(unreduced_count, 1u);
            }
        }
        store_elem<N>(store, ld.slot, lane, g.log2_wt, v);
        if (rawflag) rawflag[((tid >> g.log2_wt) << g.log2_wt) + lane] = raw_ge_p;
    }
}

// Gates that are rare on the arithmetic path; they run in their own kernel (k_level<N, true>) so the
// hot ADD/MUL kernel stays small.  A level's ops are opcode-sorted, so the split is two sub-ranges.
//   AND / XOR act on canonical residues (evaluator.rs:924-930): leave Montgomery form, operate, re-enter.
//   NOT is (a == 0) ? 1 : 0 (evaluator.rs:932-938); zero is zero in Montgomery form too.
//   ASSERT passes the operand through so the caller tests it.
// and / xor with an operand the reference holds UNREDUCED (an instance / witness / constant value >= p feeding the gate
// directly): (a & b) % m and (a ^ b) % m on the raw integers (evaluator.rs:924-930).  The raw bytes are still resident
// (d_inst / d_wit, the raw constant table); the other operand is its canonical residue.  The result is reduced by Horner
// over element-sized chunks from the top, like the input kernel does for wide values.  Rare: kept out of line.
template <int N>
__device__ __noinline__ void bitwise_raw(uint32_t* r, const uint32_t* a, const uint32_t* b, bool is_and, bool fa, bool fb, uint32_t slot_a,
                                         uint32_t slot_b, uint32_t widx, const RawCtx& rc, const FieldParams& fp) {
    const uint8_t* src[2] = {nullptr, nullptr};
    uint32_t len[2] = {0, 0};
    const uint32_t slot[2] = {slot_a, slot_b};
    const bool flagged[2] = {fa, fb};
    uint32_t canon[2][N], one[N];
#pragma unroll
    for (int k = 0; k < N; k++) one[k] = (k == 0);
    uint32_t n_chunks = 1;
    for (int o = 0; o < 2; o++) {
        if (flagged[o]) {
            const InputLoad ld = rc.loads[slot[o]];
            if (ld.kind == V_CONST) {
                src[o] = rc.const_raw + (size_t)ld.index * rc.const_raw_stride;
                len[o] = rc.const_raw_stride;
            } else {
                src[o] = (ld.kind == V_INSTANCE ? rc.in.inst + (uint64_t)widx * rc.in.inst_set_stride
                                                : rc.in.wit + (uint64_t)widx * rc.in.wit_set_stride) + (uint64_t)ld.index * rc.in.stride;
                len[o] = rc.in.stride;
            }
            n_chunks = max(n_chunks, (len[o] + 4 * N - 1) / (4 * N));
        } else {
            fe_mont_mul<N>(canon[o], o == 0 ? a : b, one, fp.p, fp.n0inv);
        }
    }
    uint32_t acc[N];
#pragma unroll
    for (int k = 0; k < N; k++) acc[k] = 0;
    for (uint32_t c = n_chunks; c-- > 0;) {
        uint32_t v[2][N];
        for (int o = 0; o < 2; o++) {
#pragma unroll
            for (int k = 0; k < N; k++) v[o][k] = (!flagged[o] && c == 0) ? canon[o][k] : 0u;
            if (flagged[o]) {
                const uint32_t b0 = c * 4 * N;
                for (uint32_t q = 0; q < 4 * N && b0 + q < len[o]; q++) v[o][q >> 2] |= (uint32_t)src[o][b0 + q] << (8 * (q & 3));
            }
        }
        uint32_t x[N], m[N], t[N];
#pragma unroll
        for (int k = 0; k < N; k++) x[k] = is_and ? (v[0][k] & v[1][k]) : (v[0][k] ^ v[1][k]);
        fe_mont_mul<N>(m, x, fp.r2, fp.p, fp.n0inv);  // x * R mod p, for any N-limb x
        if (c + 1 < n_chunks) {
            fe_mont_mul<N>(t, acc, fp.r2, fp.p, fp.n0inv);
            fe_add<N>(acc, t, m, fp.p);
        } else {
#pragma unroll
            for (int k = 0; k < N; k++) acc[k] = m[k];
        }
    }
#pragma unroll
    for (int k = 0; k < N; k++) r[k] = acc[k];
}

template <int N>
__device__ __forceinline__ void rare_gate(uint32_t* r, const uint32_t* a, const uint32_t* b, const uint4& d, uint32_t lane, const TileGeom& g,
                                          const RawCtx& rc, const FieldParams& fp) {
    const uint32_t opc = d.w & 0xff;
    // the "raw integer >= p" flags of the operands that are input values (F_RAW: a, F_RAWB: b)
    const bool fa = (d.w & F_RAW) && rc.rawflag != nullptr && rc.rawflag[((size_t)d.x << g.log2_wt) + lane] != 0;
    if (opc == D_AND || opc == D_XOR) {
        const bool fb = (d.w & F_RAWB) && rc.rawflag != nullptr && rc.rawflag[((size_t)d.y << g.log2_wt) + lane] != 0;
        if (fa || fb) {
            bitwise_raw<N>(r, a, b, opc == D_AND, fa, fb, d.x, d.y, g.batch0 + lane, rc, fp);
            return;
        }
        uint32_t one[N], ca[N], cb[N], x[N];
#pragma unroll
        for (int k = 0; k < N; k++) one[k] = (k == 0);
        fe_mont_mul<N>(ca, a, one, fp.p, fp.n0inv);
        fe_mont_mul<N>(cb, b, one, fp.p, fp.n0inv);
        if (opc == D_AND) fe_and_canon<N>(x, ca, cb);
        else fe_xor_canon<N>(x, ca, cb, fp.p);
        fe_mont_mul<N>(r, x, fp.r2, fp.p, fp.n0inv);
    } else if (opc == D_NOT) {
        bool z = fe_is_zero<N>(a) && !fa;  // an input >= p is a non-zero integer even when it is 0 mod p
#pragma unroll
        for (int k = 0; k < N; k++) r[k] = z ? fp.one[k] : 0u;
    } else {  // standalone assertion on an input: report non-zero when the raw integer is (evaluator.rs:900-906)
#pragma unroll
        for (int k = 0; k < N; k++) r[k] = a[k];
        if (fa) r[0] |= 1u;
    }
}

// ---------------------------------------------------------------------------------------------
// one wavefront of gates for one tile of witnesses
// thread <-> (gate, witness lane); lane is the fast index, so a warp works on ONE gate for 32
// consecutive witnesses whenever the tile holds >= 32 witnesses (no divergence, coalesced rows).
// ---------------------------------------------------------------------------------------------
template <int N, bool RARE>
__global__ void __launch_bounds__(256)
k_level(const GateOp* __restrict__ ops, const uint32_t* __restrict__ aseq, uint64_t n_ops, uint32_t* __restrict__ store,
        const uint32_t* __restrict__ consts_mont, uint32_t* __restrict__ first_fail, RawCtx rc, TileGeom g, FieldParams fp) {
    const uint64_t total = n_ops << g.log2_wt;
    const uint32_t wt_mask = (1u << g.log2_wt) - 1;
    const bool single = g.log2_wt == 0;
    for (uint64_t tid = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; tid < total;
         tid += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t lane = (uint32_t)tid & wt_mask;
        const uint64_t gi = tid >> g.log2_wt;
        const uint4 raw = __ldg(reinterpret_cast<const uint4*>(ops) + gi);
        const uint32_t opc = raw.w & 0xff;
        uint32_t a[N], b[N], r[N];
        load_elem<N>(a, store, raw.x, lane, g.log2_wt);
        // second operand: a wire (ADD/MUL/AND/XOR) or an entry of the Montgomery constant table
        if (!RARE) {
            if (opc == D_ADDC || opc == D_MULC) {
#pragma unroll
                for (int k = 0; k < N; k++) b[k] = __ldg(consts_mont + (size_t)raw.y * N + k);
            } else {
                load_elem<N>(b, store, raw.y, lane, g.log2_wt);
            }
            if (opc == D_ADD || opc == D_ADDC) fe_add<N>(r, a, b, fp.p);
            else fe_mont_mul<N>(r, a, b, fp.p, fp.n0inv);
        } else {
            if (opc == D_AND || opc == D_XOR) {
                load_elem<N>(b, store, raw.y, lane, g.log2_wt);
            } else {
#pragma unroll
                for (int k = 0; k < N; k++) b[k] = 0;
            }
            rare_gate<N>(r, a, b, raw, lane, g, rc, fp);
        }
        if (!(raw.w & (F_NOSTORE | g.skip_mask))) store_elem<N>(store, raw.z, lane, g.log2_wt, r);
        if (raw.w & F_ASSERT) {
            bool fail = !fe_is_zero<N>(r) && lane < g.n_valid;
            report_fail(fail, __ldg(aseq + gi), first_fail, g.batch0 + lane, single);
        }
    }
}

// Software-pipelined variant of the hot kernel: the gate descriptor is fetched two iterations ahead and the
// operand limbs one iteration ahead, so a thread always has the next gate's 4 x 16-byte loads in flight
// while it runs the current gate's integer chain (the dependent descriptor -> operand latency and the
// compute phase no longer serialise with the memory phase).
// LPT = witness lanes per thread.  For the narrow fields (N = 1, 2 limbs) a thread takes 4 / 2 adjacent lanes: their
// elements are adjacent in the wire store (witness-minor layout), so one 16-byte vector load brings them all and a
// warp still moves 512 bytes per request — the "packed element" of LPT * N limbs is addressed exactly like a 4-limb
// element of a tile with Wt / LPT lanes.  LPT = 1 for N >= 4.
template <int N, int LPT>
__device__ __forceinline__ void load_operands(uint32_t* a, uint32_t* b, const uint4& d, const uint32_t* __restrict__ store,
                                              const uint32_t* __restrict__ consts_mont, uint32_t plane, uint32_t log2_pwt) {
    constexpr int PN = N * LPT;
    const uint32_t opc = d.w & 0xff;
    load_elem<PN>(a, store, d.x, plane, log2_pwt);
    if (opc == D_ADDC || opc == D_MULC) {
#pragma unroll
        for (int l = 0; l < LPT; l++)
#pragma unroll
            for (int k = 0; k < N; k++) b[l * N + k] = __ldg(consts_mont + (size_t)d.y * N + k);
    } else {
        load_elem<PN>(b, store, d.y, plane, log2_pwt);
    }
}

#ifndef ZKB_LEVEL_PIPE_MIN_CTAS
#define ZKB_LEVEL_PIPE_MIN_CTAS 4  // 64 registers: 4 resident CTAs per SM measured 6 % faster than 3 (scripts/ab_min_ctas.sh)
#endif
template <int N, int LPT, uint32_t FORM = kMulFormGeneric>
__global__ void __launch_bounds__(256, ZKB_LEVEL_PIPE_MIN_CTAS)
k_level_pipe(const GateOp* __restrict__ ops, const uint32_t* __restrict__ aseq, uint64_t n_ops, uint32_t* __restrict__ store,
             const uint32_t* __restrict__ consts_mont, uint32_t* __restrict__ first_fail, TileGeom g, FieldParams fp) {
    constexpr int PN = N * LPT;
    constexpr uint32_t kLog2Lpt = LPT == 4 ? 2 : LPT == 2 ? 1 : 0;
    const uint32_t log2_pwt = g.log2_wt - kLog2Lpt;  // packed lanes per tile
    const uint64_t total = n_ops << log2_pwt;
    const uint32_t pwt_mask = (1u << log2_pwt) - 1;
    const bool single = g.log2_wt == 0;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    uint64_t t0 = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (t0 >= total) return;
    const uint4* dptr = reinterpret_cast<const uint4*>(ops);
    uint64_t t1 = t0 + stride, t2 = t1 + stride;
    uint4 d0 = __ldg(dptr + (t0 >> log2_pwt));
    uint4 d1 = t1 < total ? __ldg(dptr + (t1 >> log2_pwt)) : make_uint4(0, 0, 0, 0);
    uint32_t a0[PN], b0[PN], a1[PN], b1[PN];
    load_operands<N, LPT>(a0, b0, d0, store, consts_mont, (uint32_t)t0 & pwt_mask, log2_pwt);
    while (true) {
        uint4 d2 = make_uint4(0, 0, 0, 0);
        if (t2 < total) d2 = __ldg(dptr + (t2 >> log2_pwt));
        const bool more = t1 < total;
        if (more) load_operands<N, LPT>(a1, b1, d1, store, consts_mont, (uint32_t)t1 & pwt_mask, log2_pwt);
        // ---- current gate ----
        const uint32_t opc = d0.w & 0xff;
        const uint32_t plane = (uint32_t)t0 & pwt_mask;
        uint32_t r[PN];
#pragma unroll
        for (int l = 0; l < LPT; l++) {
            if (opc == D_ADD || opc == D_ADDC) fe_add<N>(r + l * N, a0 + l * N, b0 + l * N, fp.p);
            else fe_mont_mul_form<N, FORM>(r + l * N, a0 + l * N, b0 + l * N, fp.p, fp.n0inv);
        }
        if (!(d0.w & (F_NOSTORE | g.skip_mask))) store_elem<PN>(store, d0.z, plane, log2_pwt, r);
        if (d0.w & F_ASSERT) {
            const uint32_t seq = __ldg(aseq + (t0 >> log2_pwt));
#pragma unroll
            for (int l = 0; l < LPT; l++) {
                const uint32_t lane = plane * LPT + l;
                bool fail = !fe_is_zero<N>(r + l * N) && lane < g.n_valid;
                report_fail(fail, seq, first_fail, g.batch0 + lane, single);
            }
        }
        if (!more) break;
#pragma unroll
        for (int k = 0; k < PN; k++) {
            a0[k] = a1[k];
            b0[k] = b1[k];
        }
        d0 = d1;
        d1 = d2;
        t0 = t1;
        t1 = t2;
        t2 += stride;
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// k_level_tma: the same wavefront step with the operand rows brought in by the bulk-copy engine (cp.async.bulk, 1-D TMA)
// instead of per-thread vector loads.  In the witness-minor layout a gate's operand for a block of 256 lanes is two
// contiguous 4 KB pieces (N = 8: one per 16-byte chunk row; adjacent, i.e. one 8 KB block, when the tile is 256 lanes
// wide), so a CTA <-> one (gate, lane block) per iteration: one elected thread arms an mbarrier with the byte count and
// issues the bulk copies into a ring of STAGES shared-memory stages, STAGES items ahead; all 256 threads wait on the
// stage's mbarrier, take their two 16-byte chunks per operand from shared memory (conflict-free: consecutive lanes,
// consecutive 16-byte words), and the stage is handed back after one block barrier.  Results leave with plain 16-byte
// vector stores (each warp writes 512 contiguous bytes already).
// For 8-limb fields and tiles of >= 256 lanes (the headline configuration); everything else runs k_level_pipe.
// Measured on the headline shape (scripts/ab_level_tma*.sh, profiles/r02g_ab_level_tma*.log): 73.4-74.2 G gate-evals/s against
// 69.3-69.6 for k_level_pipe on the same box, i.e. 1.01-1.02 x the measured copy peak; bulk STORES of the results through shared memory on top changed
// nothing (77.6 vs 77.4 on one box, scripts/ab_level_tma3.sh at commit time) and were dropped.  ZKB_LEVEL_TMA=0 switches back to k_level_pipe.
// ---------------------------------------------------------------------------------------------------------------------
#ifndef ZKB_TMA_STAGES
#define ZKB_TMA_STAGES 3
#endif
#ifndef ZKB_TMA_MIN_CTAS
#define ZKB_TMA_MIN_CTAS 4
#endif
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src), "r"(bytes),
                 "r"(bar)
                 : "memory");
}
__device__ __forceinline__ uint4 lds128(uint32_t a) {
    uint4 v;
    asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a));
    return v;
}

constexpr size_t kTmaSmemBytes = (size_t)ZKB_TMA_STAGES * 16384;

template <int N, uint32_t FORM>
__global__ void __launch_bounds__(256, ZKB_TMA_MIN_CTAS)
k_level_tma(const GateOp* __restrict__ ops, const uint32_t* __restrict__ aseq, uint64_t n_ops, uint32_t* __restrict__ store,
            const uint32_t* __restrict__ consts_mont, uint32_t* __restrict__ first_fail, TileGeom g, FieldParams fp) {
    static_assert(N == 8, "two 16-byte chunks per element");
    constexpr int S = ZKB_TMA_STAGES;
    constexpr uint32_t ELEM = 8192, STAGE = 2 * ELEM;
    extern __shared__ __align__(128) uint8_t tma_smem[];
    __shared__ __align__(8) uint64_t full_bar[S];
    const uint32_t smem0 = (uint32_t)__cvta_generic_to_shared(tma_smem);
    const uint32_t bar0 = (uint32_t)__cvta_generic_to_shared(full_bar);
    const uint4* dptr = reinterpret_cast<const uint4*>(ops);
    const uint8_t* store_b = reinterpret_cast<const uint8_t*>(store);
    // item = (gate, block of 256 lanes): a tile of 2^log2_wt lanes holds 2^(log2_wt - 8) blocks; the two 16-byte chunks of an
    // element are rows of 16 << log2_wt bytes, 4 KB of each belong to a block (adjacent when the tile IS one block)
    const uint32_t log2_q = g.log2_wt - 8;
    const uint32_t q_mask = (1u << log2_q) - 1;
    const uint64_t n_items = n_ops << log2_q;
    const uint32_t row = 4096u << log2_q;  // bytes between the chunk rows of one element
    const uint64_t stride = gridDim.x;
    uint64_t gi = blockIdx.x;
    if (gi >= n_items) return;
    auto issue = [&](uint32_t stage, const uint4& d, uint32_t q) {  // elected thread: arm the stage's barrier, start the copies
        const uint32_t opc = d.w & 0xff;
        const bool two = !(opc == D_ADDC || opc == D_MULC);
        const uint32_t bar = bar0 + stage * 8;
        mbar_expect_tx(bar, two ? STAGE : ELEM);
        const uint8_t* pa = store_b + (size_t)d.x * 2 * row + (size_t)q * 4096;
        bulk_g2s(smem0 + stage * STAGE, pa, 4096, bar);
        bulk_g2s(smem0 + stage * STAGE + 4096, pa + row, 4096, bar);
        if (two) {
            const uint8_t* pb = store_b + (size_t)d.y * 2 * row + (size_t)q * 4096;
            bulk_g2s(smem0 + stage * STAGE + ELEM, pb, 4096, bar);
            bulk_g2s(smem0 + stage * STAGE + ELEM + 4096, pb + row, 4096, bar);
        }
    };
    uint64_t gp = gi;  // producer cursor (thread 0): next gate to request
    uint4 dp = make_uint4(0, 0, 0, 0);
    if (threadIdx.x == 0) {
#pragma unroll
        for (int i = 0; i < S; i++) mbar_init(bar0 + i * 8, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
#pragma unroll
        for (int i = 0; i < S; i++) {
            if (gp < n_items) issue(i, __ldg(dptr + (gp >> log2_q)), (uint32_t)gp & q_mask);
            gp += stride;
        }
        if (gp < n_items) dp = __ldg(dptr + (gp >> log2_q));
    }
    __syncthreads();
    uint4 d0 = __ldg(dptr + (gi >> log2_q));
    for (uint32_t it = 0;; it++) {
        const uint64_t gn = gi + stride;
        uint4 d1 = make_uint4(0, 0, 0, 0);
        if (gn < n_items) d1 = __ldg(dptr + (gn >> log2_q));
        const uint32_t lane = (((uint32_t)gi & q_mask) << 8) + threadIdx.x;
        const uint32_t stage = it % S, parity = (it / S) & 1;
        const uint32_t opc = d0.w & 0xff;
        uint32_t a[N], b[N], r[N];
        mbar_wait(bar0 + stage * 8, parity);
        const uint32_t sa = smem0 + stage * STAGE + threadIdx.x * 16;
        unpack(lds128(sa), a);
        unpack(lds128(sa + 4096), a + 4);
        if (opc == D_ADDC || opc == D_MULC) {
#pragma unroll
            for (int k = 0; k < N; k++) b[k] = __ldg(consts_mont + (size_t)d0.y * N + k);
        } else {
            unpack(lds128(sa + ELEM), b);
            unpack(lds128(sa + ELEM + 4096), b + 4);
        }
        __syncthreads();  // every thread holds its limbs: the stage can be refilled
        if (threadIdx.x == 0) {
            if (gp < n_items) {
                issue(stage, dp, (uint32_t)gp & q_mask);
                gp += stride;
                if (gp < n_items) dp = __ldg(dptr + (gp >> log2_q));
            }
        }
        if (opc == D_ADD || opc == D_ADDC) fe_add<N>(r, a, b, fp.p);
        else fe_mont_mul_form<N, FORM>(r, a, b, fp.p, fp.n0inv);
        if (!(d0.w & (F_NOSTORE | g.skip_mask))) store_elem<N>(store, d0.z, lane, g.log2_wt, r);
        if (d0.w & F_ASSERT) {
            const uint32_t seq = __ldg(aseq + (gi >> log2_q));
            bool fail = !fe_is_zero<N>(r) && lane < g.n_valid;
            report_fail(fail, seq, first_fail, g.batch0 + lane, false);
        }
        if (gn >= n_items) break;
        d0 = d1;
        gi = gn;
    }
}

// Grid barrier on one monotonic counter (per context, never reset: the host hands every launch its starting value).
// A CTA arrives with one red.release.gpu after its block barrier and polls the counter until all have.  Measured SLOWER than
// cooperative_groups' grid.sync() (zkb_debug_barrier_cost, profiles/r02h_ab_c2.log): opt-in only (ZKB_COUNTER_BARRIER=1).
// All CTAs must be resident: the kernel is still launched with cudaLaunchCooperativeKernel.
__device__ __forceinline__ void grid_barrier(uint32_t* ctr, uint32_t target) {
    __syncthreads();
    if (threadIdx.x == 0) {
        asm volatile("red.release.gpu.global.add.u32 [%0], 1;" ::"l"(ctr) : "memory");
        uint32_t v;
        do {  // relaxed polls (an acquire load is a load plus a fence, every time round), one fence once the count is there
            asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(ctr) : "memory");
        } while ((int32_t)(v - target) < 0);
        asm volatile("fence.acq_rel.gpu;" ::: "memory");
    }
    __syncthreads();
}

// All wavefronts in ONE cooperative launch, a grid barrier between levels.  For programs whose levels are
// too small to fill the chip (single-witness statements, deep narrow circuits) the per-level launch latency
// (~4-5 us) dominates; a grid.sync() costs ~1-2 us.  Operands are read with ld.global.cg because they were
// written by other SMs earlier in this same launch.
// CLUSTER = true: the same loop for programs so narrow that ONE thread-block cluster (8 CTAs on neighbouring SMs of
// one die) holds a whole wavefront: the barrier between levels is the hardware cluster barrier (barrier.cluster
// arrive.release / wait.acquire, ~0.2 us) instead of a grid barrier through L2 atomics.
#ifdef ZKB_COOP_PROFILE
__device__ __forceinline__ long long zkb_clock() {  // clock read that memory operations are not moved across
    long long t;
    asm volatile("mov.u64 %0, %%clock64;" : "=l"(t)::"memory");
    return t;
}
#endif
// A descriptor load that stays where it is written: a plain __ldg of __restrict__ data is an invariant load, which the
// compiler is free to sink below the barrier down to its first use, putting the memory latency back on the critical path.
__device__ __forceinline__ uint4 ldg_pinned(const uint4* p) {
    uint4 v;
    asm volatile("ld.global.nc.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
    return v;
}

template <int N, bool CLUSTER>
__global__ void __launch_bounds__(CLUSTER ? 512 : 256)
k_levels_coop(const GateOp* __restrict__ ops, const uint32_t* __restrict__ aseq, const uint64_t* __restrict__ level_off,
              uint32_t n_levels, uint32_t* store, const uint32_t* __restrict__ consts_mont, uint32_t* __restrict__ first_fail,
              RawCtx rc, TileGeom g, FieldParams fp, uint32_t* barrier_ctr, uint32_t barrier_base) {
    const uint32_t wt_mask = (1u << g.log2_wt) - 1;
    const bool single = g.log2_wt == 0;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;  // CLUSTER: the grid is exactly one cluster
    const uint64_t tid0 = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    const uint4* dptr = reinterpret_cast<const uint4*>(ops);
    // wavefront boundaries from shared memory: the barriers flush L1, a global read of level_off[l + 2] would be one L2
    // round trip at the top of every level, in front of the descriptor prefetch that needs it
    constexpr uint32_t kOffCache = 2048;
    __shared__ uint64_t s_off[kOffCache + 1];
    for (uint32_t i = threadIdx.x; i <= n_levels && i <= kOffCache; i += blockDim.x) s_off[i] = level_off[i];
    __syncthreads();
    auto off = [&](uint32_t i) -> uint64_t { return i <= kOffCache ? s_off[i] : level_off[i]; };
    // the first descriptor of each level is fetched BEFORE the barrier that precedes the level (descriptors
    // do not depend on wire data), taking one memory latency off the per-level critical path
    uint64_t lo = off(0), hi = n_levels ? off(1) : lo;
    uint4 first = make_uint4(0, 0, 0, 0);
    if (tid0 < ((hi - lo) << g.log2_wt)) first = ldg_pinned(dptr + lo + (tid0 >> g.log2_wt));
#ifdef ZKB_COOP_PROFILE
    long long prof[7] = {0, 0, 0, 0, 0, 0, 0};
#endif
    for (uint32_t l = 0; l < n_levels; l++) {
#ifdef ZKB_COOP_PROFILE
        const long long th0 = zkb_clock();
#endif
        const uint64_t total = (hi - lo) << g.log2_wt;
        uint64_t nlo = hi, nhi = hi;
        uint4 next_first = make_uint4(0, 0, 0, 0);
        if (l + 1 < n_levels) {
            nhi = off(l + 2);
            if (tid0 < ((nhi - nlo) << g.log2_wt)) next_first = ldg_pinned(dptr + nlo + (tid0 >> g.log2_wt));
        }
#ifdef ZKB_COOP_PROFILE
        const long long tw0 = zkb_clock();
        prof[0] += tw0 - th0;
#endif
        for (uint64_t tid = tid0; tid < total; tid += stride) {
            const uint32_t lane = (uint32_t)tid & wt_mask;
            const uint64_t gi = lo + (tid >> g.log2_wt);
            const uint4 raw = tid == tid0 ? first : __ldg(dptr + gi);
            const uint32_t opc = raw.w & 0xff;
            uint32_t a[N], b[N], r[N];
            load_elem_coherent<N>(a, store, raw.x, lane, g.log2_wt);
            if (opc == D_ADDC || opc == D_MULC) {
#pragma unroll
                for (int k = 0; k < N; k++) b[k] = __ldg(consts_mont + (size_t)raw.y * N + k);
            } else if (opc == D_ADD || opc == D_MUL || opc == D_AND || opc == D_XOR) {
                load_elem_coherent<N>(b, store, raw.y, lane, g.log2_wt);
            } else {
#pragma unroll
                for (int k = 0; k < N; k++) b[k] = 0;
            }
#ifdef ZKB_COOP_PROFILE
            long long tq0 = zkb_clock();
            prof[6] += tq0 - tw0;
            if ((a[0] ^ b[0]) == 0x12345678u) tq0++;  // waits for the operands
            const long long tq1 = zkb_clock();
            prof[3] += tq1 - tq0;
#endif
            if (opc == D_ADD || opc == D_ADDC) fe_add<N>(r, a, b, fp.p);
            else if (opc == D_MUL || opc == D_MULC) fe_mont_mul<N>(r, a, b, fp.p, fp.n0inv);
            else rare_gate<N>(r, a, b, raw, lane, g, rc, fp);
#ifdef ZKB_COOP_PROFILE
            long long tq2 = zkb_clock();
            if (r[0] == 0x12345679u) tq2++;
            prof[4] += tq2 - tq1;
#endif
            if (!(raw.w & F_NOSTORE)) store_elem<N>(store, raw.z, lane, g.log2_wt, r);
            if (raw.w & F_ASSERT) {
                bool fail = !fe_is_zero<N>(r) && lane < g.n_valid;
                report_fail(fail, __ldg(aseq + gi), first_fail, g.batch0 + lane, single);
            }
#ifdef ZKB_COOP_PROFILE
            prof[5] += zkb_clock() - tq2;
#endif
        }
#ifdef ZKB_COOP_PROFILE
        prof[1] += zkb_clock() - tw0;
#endif
        first = next_first;
        lo = nlo;
        hi = nhi;
        if (l + 1 < n_levels) {
#ifdef ZKB_COOP_PROFILE
            const long long tb0 = zkb_clock();
#endif
            if (CLUSTER) cg::this_cluster().sync();
            else if (barrier_ctr) grid_barrier(barrier_ctr, barrier_base + gridDim.x * (l + 1));
            else cg::this_grid().sync();
#ifdef ZKB_COOP_PROFILE
            prof[2] += zkb_clock() - tb0;
#endif
        }
    }
#ifdef ZKB_COOP_PROFILE
    if ((threadIdx.x & 31) == 0 && (blockIdx.x == 0 || blockIdx.x == gridDim.x - 1) && (threadIdx.x == 0 || threadIdx.x == blockDim.x - 32))
        printf("coop profile cta %u warp %u: levels %u  head %lld  work %lld (issue %lld operands %lld compute %lld store+assert %lld)  barrier %lld  (cycles per level)\n",
               blockIdx.x, threadIdx.x / 32, n_levels, prof[0] / n_levels, prof[1] / n_levels, prof[6] / n_levels, prof[3] / n_levels, prof[4] / n_levels,
               prof[5] / n_levels, prof[2] / n_levels);
#endif
}

// ---------------------------------------------------------------------------------------------------------------------
// k_levels_flow: every wavefront in ONE cooperative launch and NO barrier at all — dataflow.  For one witness over a 1- or
// 2-limb field an element is one naturally aligned 4- / 8-byte word, and the all-ones word is no residue (a stored value is
// < p <= 2^(32N) - 1): it marks "not computed yet".  The host fills the computed slots with it before the launch; a gate
// polls its operand words (ld.relaxed.gpu: single-copy atomic, served by L2) until they are values, computes, and publishes
// its result with one st.relaxed.gpu — the value IS the flag, so a producer-consumer hop costs one L2 round trip instead of
// store -> fence -> grid barrier (1.2 us) -> descriptor -> gather (C2: 4.5 us per wavefront, DESIGN.md section 5).
// Progress: all CTAs are resident (cooperative launch) and every thread walks its gates wavefront by wavefront, so the
// lowest wavefront with an unfinished gate only waits on finished ones.  Inside one loop trip the lanes of a warp hold gates
// of the SAME wavefront (the stride loop restarts at every wavefront boundary): lanes never wait on each other, which matters
// because the compiler reconverges the warp after the polling loop.  Needs a plan without slot re-use (a slot written twice
// would make a late reader of the first value see the second).
// ---------------------------------------------------------------------------------------------------------------------
// one poll of an element's word: all ones = not computed yet
template <int N>
__device__ __forceinline__ uint64_t flow_peek(const uint32_t* store, uint32_t slot) {
    if constexpr (N == 2) {
        uint64_t v;
        asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(reinterpret_cast<const uint64_t*>(store) + slot) : "memory");
        return v;
    } else {
        uint32_t v;
        asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(store + slot) : "memory");
        return v == ~0u ? ~0ull : (uint64_t)v;
    }
}
template <int N>
__device__ __forceinline__ void flow_publish_elem(uint32_t* store, uint32_t slot, const uint32_t* r) {
    if constexpr (N == 2) {
        const uint64_t v = (uint64_t)r[1] << 32 | r[0];
        asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(reinterpret_cast<uint64_t*>(store) + slot), "l"(v) : "memory");
    } else {
        asm volatile("st.relaxed.gpu.global.u32 [%0], %1;" ::"l"(store + slot), "r"(r[0]) : "memory");
    }
}

template <int N>
__global__ void __launch_bounds__(256)
k_levels_flow(const GateOp* __restrict__ ops, const uint32_t* __restrict__ aseq, const uint64_t* __restrict__ level_off,
              uint32_t n_levels, uint32_t* store, const uint32_t* __restrict__ consts_mont, uint32_t* __restrict__ first_fail,
              RawCtx rc, TileGeom g, FieldParams fp, uint32_t sleep_ns) {
    static_assert(N <= 2, "one word per element");
    constexpr uint32_t kOffCache = 2048;
    __shared__ uint64_t s_off[kOffCache + 1];
    for (uint32_t i = threadIdx.x; i <= n_levels && i <= kOffCache; i += blockDim.x) s_off[i] = level_off[i];
    __syncthreads();
    auto off = [&](uint32_t i) -> uint64_t { return i <= kOffCache ? s_off[i] : level_off[i]; };
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    const uint64_t tid0 = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    const uint4* dptr = reinterpret_cast<const uint4*>(ops);
    // the descriptor of a thread's first gate of the NEXT wavefront is fetched while it works on (waits in) the current one:
    // descriptors do not depend on wire data, and the fetch would otherwise head every hop of the dependency chain
    uint4 first = make_uint4(0, 0, 0, 0);
    if (n_levels && off(0) + tid0 < off(1)) first = ldg_pinned(dptr + off(0) + tid0);
    for (uint32_t l = 0; l < n_levels; l++) {
        const uint64_t lo = off(l), hi = off(l + 1);
        uint4 next_first = make_uint4(0, 0, 0, 0);
        if (l + 1 < n_levels && hi + tid0 < off(l + 2)) next_first = ldg_pinned(dptr + hi + tid0);
        for (uint64_t gi = lo + tid0; gi < hi; gi += stride) {
            const uint4 raw = gi == lo + tid0 ? first : __ldg(dptr + gi);
            const uint32_t opc = raw.w & 0xff;
            const bool two = opc == D_ADD || opc == D_MUL || opc == D_AND || opc == D_XOR;
            uint32_t a[N], b[N], r[N];
            // both operand polls in flight together
            uint64_t va = flow_peek<N>(store, raw.x);
            uint64_t vb = two ? flow_peek<N>(store, raw.y) : 0;
            while (va == ~0ull) {
                if (sleep_ns) __nanosleep(sleep_ns);
                va = flow_peek<N>(store, raw.x);
            }
            while (vb == ~0ull) {
                if (sleep_ns) __nanosleep(sleep_ns);
                vb = flow_peek<N>(store, raw.y);
            }
            a[0] = (uint32_t)va;
            if constexpr (N == 2) a[1] = (uint32_t)(va >> 32);
            if (opc == D_ADDC || opc == D_MULC) {
#pragma unroll
                for (int k = 0; k < N; k++) b[k] = __ldg(consts_mont + (size_t)raw.y * N + k);
            } else {
                b[0] = (uint32_t)vb;
                if constexpr (N == 2) b[1] = (uint32_t)(vb >> 32);
            }
            if (opc == D_ADD || opc == D_ADDC) fe_add<N>(r, a, b, fp.p);
            else if (opc == D_MUL || opc == D_MULC) fe_mont_mul<N>(r, a, b, fp.p, fp.n0inv);
            else rare_gate<N>(r, a, b, raw, 0u, g, rc, fp);
            if (!(raw.w & F_NOSTORE)) flow_publish_elem<N>(store, raw.z, r);
            if ((raw.w & F_ASSERT) && !fe_is_zero<N>(r)) atomicMin(first_fail + g.batch0, __ldg(aseq + gi));
        }
        first = next_first;
        // the warp moves on together: a lane without a gate in this wavefront must not run ahead and poll for a value that a
        // lane of its own warp has yet to produce (divergent lanes of one warp share its issue slot)
        __syncwarp();
    }
}

// The same dataflow launch for elements wider than one atomic word (4- and 8-limb fields): a flag word per slot carries the
// number of the run that produced the value (never reset: a new run is a new number).  Producer: value stores, fence, flag
// store; consumer: relaxed polls of both operands' flags, one fence, then the limb loads (L2-coherent).  A hop costs a flag
// round trip plus a value round trip instead of one, still without any barrier.  Slots below n_ready hold level-0 values
// (inputs, group outputs) written by earlier kernels of the stream.
template <int N>
__global__ void __launch_bounds__(256)
k_levels_flow_wide(const GateOp* __restrict__ ops, const uint32_t* __restrict__ aseq, const uint64_t* __restrict__ level_off,
                   uint32_t n_levels, uint32_t* store, const uint32_t* __restrict__ consts_mont, uint32_t* __restrict__ first_fail,
                   RawCtx rc, TileGeom g, FieldParams fp, uint32_t* flags, uint32_t epoch, uint32_t n_ready) {
    constexpr uint32_t kOffCache = 2048;
    __shared__ uint64_t s_off[kOffCache + 1];
    for (uint32_t i = threadIdx.x; i <= n_levels && i <= kOffCache; i += blockDim.x) s_off[i] = level_off[i];
    __syncthreads();
    auto off = [&](uint32_t i) -> uint64_t { return i <= kOffCache ? s_off[i] : level_off[i]; };
    auto peek = [&](uint32_t slot) -> bool {
        if (slot < n_ready) return true;
        uint32_t v;
        asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(flags + slot) : "memory");
        return v == epoch;
    };
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    const uint64_t tid0 = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    const uint4* dptr = reinterpret_cast<const uint4*>(ops);
    uint4 first = make_uint4(0, 0, 0, 0);
    if (n_levels && off(0) + tid0 < off(1)) first = ldg_pinned(dptr + off(0) + tid0);
    for (uint32_t l = 0; l < n_levels; l++) {
        const uint64_t lo = off(l), hi = off(l + 1);
        uint4 next_first = make_uint4(0, 0, 0, 0);
        if (l + 1 < n_levels && hi + tid0 < off(l + 2)) next_first = ldg_pinned(dptr + hi + tid0);
        for (uint64_t gi = lo + tid0; gi < hi; gi += stride) {
            const uint4 raw = gi == lo + tid0 ? first : __ldg(dptr + gi);
            const uint32_t opc = raw.w & 0xff;
            const bool two = opc == D_ADD || opc == D_MUL || opc == D_AND || opc == D_XOR;
            bool ra = peek(raw.x), rb = two ? peek(raw.y) : true;
            while (!ra) ra = peek(raw.x);
            while (!rb) rb = peek(raw.y);
            asm volatile("fence.acq_rel.gpu;" ::: "memory");
            uint32_t a[N], b[N], r[N];
            load_elem_coherent<N>(a, store, raw.x, 0u, 0u);
            if (opc == D_ADDC || opc == D_MULC) {
#pragma unroll
                for (int k = 0; k < N; k++) b[k] = __ldg(consts_mont + (size_t)raw.y * N + k);
            } else if (two) {
                load_elem_coherent<N>(b, store, raw.y, 0u, 0u);
            } else {
#pragma unroll
                for (int k = 0; k < N; k++) b[k] = 0;
            }
            if (opc == D_ADD || opc == D_ADDC) fe_add<N>(r, a, b, fp.p);
            else if (opc == D_MUL || opc == D_MULC) fe_mont_mul<N>(r, a, b, fp.p, fp.n0inv);
            else rare_gate<N>(r, a, b, raw, 0u, g, rc, fp);
            if (!(raw.w & F_NOSTORE)) {
                store_elem<N>(store, raw.z, 0u, 0u, r);
                asm volatile("fence.acq_rel.gpu;" ::: "memory");
                asm volatile("st.relaxed.gpu.global.u32 [%0], %1;" ::"l"(flags + raw.z), "r"(epoch) : "memory");
            }
            if ((raw.w & F_ASSERT) && !fe_is_zero<N>(r)) atomicMin(first_fail + g.batch0, __ldg(aseq + gi));
        }
        first = next_first;
        __syncwarp();
    }
}

template <int N>
__global__ void k_read_values(const uint32_t* __restrict__ slots, uint32_t n, const uint32_t* __restrict__ store, uint32_t lane,
                              uint32_t log2_wt, uint32_t* __restrict__ out, FieldParams fp) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t a[N], one[N], r[N];
    load_elem<N>(a, store, slots[i], lane, log2_wt);
#pragma unroll
    for (int k = 0; k < N; k++) one[k] = (k == 0);
    fe_mont_mul<N>(r, a, one, fp.p, fp.n0inv);  // leave Montgomery form: canonical residue
#pragma unroll
    for (int k = 0; k < N; k++) out[(size_t)i * N + k] = r[k];
}

// ---------------------------------------------------------------------------------------------
// p = 2, bit-sliced: word w of slot s holds witnesses 32w .. 32w+31
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
k_bool_load_inputs(const InputLoad* __restrict__ loads, uint32_t n_loads, uint32_t* __restrict__ store,
                   const uint32_t* __restrict__ const_bits, InputDesc in, TileGeom g, uint32_t* unreduced_count,
                   uint8_t* __restrict__ rawflag, const uint8_t* __restrict__ const_flags) {
    const uint32_t log2_words = g.log2_wt - 5;
    const uint64_t total = ((uint64_t)n_loads << g.log2_wt);  // one thread per (load, lane), ballot packs
    for (uint64_t tid = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; tid < total;
         tid += (uint64_t)gridDim.x * blockDim.x) {
        uint32_t lane = (uint32_t)tid & ((1u << g.log2_wt) - 1);
        InputLoad ld = loads[tid >> g.log2_wt];
        uint32_t bit = 0;
        bool raw_ge_p = false;
        if (lane < g.n_valid) {
            if (ld.kind == V_CONST) {
                bit = const_bits[ld.index] & 1;
                raw_ge_p = const_flags != nullptr && const_flags[ld.index] != 0;
            } else {
                const uint8_t* src = (ld.kind == V_INSTANCE)
                                         ? in.inst + (uint64_t)(g.batch0 + lane) * in.inst_set_stride
                                         : in.wit + (uint64_t)(g.batch0 + lane) * in.wit_set_stride;
                src += (uint64_t)ld.index * in.stride;
                uint32_t hi = 0;
                for (uint32_t b = 0; b < in.stride; b++) hi |= (b == 0) ? (uint32_t)(src[0] >> 1) : (uint32_t)src[b];
                bit = src[0] & 1;
                raw_ge_p = hi != 0;
                if (hi) atomicAdd(unreduced_count, 1u);
            }
        }
        // blockDim is a multiple of 32 and total a multiple of 32: full warps only
        uint32_t word = __ballot_sync(0xFFFFFFFFu, bit);
        if ((lane & 31) == 0) store[((size_t)ld.slot << log2_words) + (lane >> 5)] = word;
        if (rawflag) rawflag[((tid >> g.log2_wt) << g.log2_wt) + lane] = raw_ge_p;
    }
}

// one 32-witness word of a Boolean gate
__device__ __forceinline__ uint32_t bool_gate_word(uint32_t opc, uint32_t a, uint32_t b, uint32_t cbit) {
    switch (opc) {
        case D_ADD:
        case D_XOR: return a ^ b;
        case D_MUL:
        case D_AND: return a & b;
        case D_ADDC: return a ^ (0u - cbit);
        case D_MULC: return a & (0u - cbit);
        case D_NOT: return ~a;
        default: return a;
    }
}

// thread <-> (gate, WPT consecutive 32-witness words).  WPT = 4 (one 16-byte vector per operand, 512 bytes per warp
// request) whenever a tile holds at least 128 witnesses; WPT = 1 for narrower tiles.
template <int WPT>
__device__ __forceinline__ void bool_level_items(const GateOp* __restrict__ ops, const uint32_t* __restrict__ aseq, uint64_t n_ops,
                                                 uint32_t* __restrict__ store, const uint32_t* __restrict__ const_bits,
                                                 uint32_t* __restrict__ first_fail, const uint8_t* __restrict__ rawflag, const TileGeom& g,
                                                 uint64_t tid0, uint64_t stride) {
    using V = typename Vec<WPT>::T;
    constexpr uint32_t kLog2Wpt = WPT == 4 ? 2 : 0;
    const uint32_t log2_words = g.log2_wt - 5;
    const uint32_t log2_vecs = log2_words - kLog2Wpt;  // vectors per slot
    const uint64_t total = n_ops << log2_vecs;
    const uint32_t vmask = (1u << log2_vecs) - 1;
    V* vstore = reinterpret_cast<V*>(store);
    for (uint64_t tid = tid0; tid < total; tid += stride) {
        const uint32_t vw = (uint32_t)tid & vmask;
        const uint64_t gi = tid >> log2_vecs;
        const uint4 raw = __ldg(reinterpret_cast<const uint4*>(ops) + gi);
        const uint32_t opc = raw.w & 0xff;
        const bool two = opc == D_ADD || opc == D_XOR || opc == D_MUL || opc == D_AND;
        uint32_t a[WPT], b[WPT], r[WPT];
        unpack(vstore[((size_t)raw.x << log2_vecs) + vw], a);
        if (two) unpack(vstore[((size_t)raw.y << log2_vecs) + vw], b);
        const uint32_t cbit = (opc == D_ADDC || opc == D_MULC) ? (__ldg(const_bits + raw.y) & 1) : 0u;
#pragma unroll
        for (int k = 0; k < WPT; k++) r[k] = bool_gate_word(opc, a[k], two ? b[k] : 0u, cbit);
        if ((raw.w & F_RAW) && rawflag != nullptr) {  // input values >= 2 are non-zero integers (trap 1)
#pragma unroll
            for (int k = 0; k < WPT; k++) {
                const uint32_t w = vw * WPT + k;
                uint32_t nz = 0;
                const uint8_t* f = rawflag + ((size_t)raw.x << g.log2_wt) + ((size_t)w << 5);
                for (int bq = 0; bq < 32; bq++) nz |= (uint32_t)(f[bq] != 0) << bq;
                if (opc == D_NOT) r[k] &= ~nz;
                else r[k] |= nz;
            }
        }
        if (!(raw.w & F_NOSTORE)) {
            V v;
            pack(v, r);
            vstore[((size_t)raw.z << log2_vecs) + vw] = v;
        }
        if (raw.w & F_ASSERT) {
#pragma unroll
            for (int k = 0; k < WPT; k++) {
                const uint32_t first_lane = (vw * WPT + k) << 5;
                uint32_t valid = g.n_valid > first_lane ? (g.n_valid - first_lane >= 32 ? 0xFFFFFFFFu : ((1u << (g.n_valid - first_lane)) - 1)) : 0u;
                uint32_t bad = r[k] & valid;
                if (bad) {
                    uint32_t seq = __ldg(aseq + gi);
                    while (bad) {
                        int bpos = __ffs(bad) - 1;
                        bad &= bad - 1;
                        atomicMin(first_fail + g.batch0 + first_lane + bpos, seq);
                    }
                }
            }
        }
    }
}
template <int WPT>
__global__ void __launch_bounds__(256)
k_bool_level(const GateOp* __restrict__ ops, const uint32_t* __restrict__ aseq, uint64_t n_ops, uint32_t* __restrict__ store,
             const uint32_t* __restrict__ const_bits, uint32_t* __restrict__ first_fail, const uint8_t* __restrict__ rawflag,
             TileGeom g) {
    bool_level_items<WPT>(ops, aseq, n_ops, store, const_bits, first_fail, rawflag, g, blockIdx.x * (uint64_t)blockDim.x + threadIdx.x,
                          (uint64_t)gridDim.x * blockDim.x);
}
// A run of consecutive wavefronts that each fit ONE CTA (the Xor chain behind C5's loops: one gate per wavefront): one launch,
// __syncthreads() between the wavefronts (one CTA: its global writes are visible to its own threads after the barrier)
// instead of one launch each.
template <int WPT>
__global__ void __launch_bounds__(256)
k_bool_levels_cta(const GateOp* __restrict__ ops, const uint32_t* __restrict__ aseq, const uint64_t* __restrict__ level_off, uint32_t n_levels,
                  uint32_t* store, const uint32_t* __restrict__ const_bits, uint32_t* __restrict__ first_fail,
                  const uint8_t* __restrict__ rawflag, TileGeom g) {
    for (uint32_t l = 0; l < n_levels; l++) {
        const uint64_t lo = level_off[l], hi = level_off[l + 1];
        bool_level_items<WPT>(ops + lo, aseq + lo, hi - lo, store, const_bits, first_fail, rawflag, g, threadIdx.x, blockDim.x);
        __syncthreads();
    }
}

// Call groups (program.h): thread <-> (call, 32-witness word).  A call's inputs are read from the wire store into a register
// file held in shared memory (register r of thread t at (r * 256 + t) * 4: conflict-free), the body of the function runs
// over it op by op — every thread of a warp interprets the same pre-decoded template (GroupOp: byte offsets + four masks
// of one bitwise form, two broadcast 16-byte loads, no branch) — and only the call's outputs go back to the wire store:
// the locals of a call never touch memory, and one 96-byte GroupDesc stands for n_calls x |body| gates instead of one
// 16-byte GateOp each.  thread -> group: a host-made hint per 128 calls, then a forward walk over first_call.
// WPT = 4 for tiles of >= 128 witnesses (a register is one 16-byte vector: one LDS.128 / STS.128 and one 512-byte warp
// request per operand, the op fetch and the loop control are shared by four words), WPT = 1 below.
// PARAM_OPS: the templates' ops travel as a kernel parameter (constant bank) when they fit: an op fetch is then an indexed
// constant load through the constant cache instead of two 16-byte loads through L1 — the kernel's busiest unit (l1tex 92 %).
constexpr uint32_t kGroupParamOps = 256;
struct GroupOpsParam {
    uint4 q[2 * kGroupParamOps];
};
template <int WPT, bool PARAM_OPS>
__global__ void __launch_bounds__(kGroupThreads)
k_bool_groups(const GroupDesc* __restrict__ descs, uint32_t n_groups, uint64_t total_calls, const GroupOp* __restrict__ gops,
              const uint32_t* __restrict__ tables, const uint32_t* __restrict__ hints, uint32_t* __restrict__ store,
              uint32_t log2_words, const __grid_constant__ GroupOpsParam pops) {
    using V = typename Vec<WPT>::T;
    constexpr uint32_t kLog2Wpt = WPT == 4 ? 2 : 0;
    constexpr uint32_t RS = kGroupThreads * 4 * WPT;  // bytes between consecutive registers of one thread
    extern __shared__ __align__(16) uint8_t s_regs[];
    uint8_t* R = s_regs + threadIdx.x * (4 * WPT);
    const uint32_t log2_vecs = log2_words - kLog2Wpt;
    const uint64_t total = total_calls << log2_vecs;
    const uint32_t vmask = (1u << log2_vecs) - 1;
    V* vstore = reinterpret_cast<V*>(store);
    for (uint64_t tid = blockIdx.x * (uint64_t)kGroupThreads + threadIdx.x; tid < total; tid += (uint64_t)gridDim.x * kGroupThreads) {
        const uint32_t call_g = (uint32_t)(tid >> log2_vecs), vw = (uint32_t)tid & vmask;
        uint32_t gi = __ldg(hints + (call_g >> kGroupHintShift));
        while (gi + 1 < n_groups && call_g >= __ldg(&descs[gi + 1].first_call)) gi++;
        const GroupDesc* d = descs + gi;
        const uint4 h0 = __ldg(reinterpret_cast<const uint4*>(d));      // tmpl_off, n_ops, n_out, n_in
        const uint4 h1 = __ldg(reinterpret_cast<const uint4*>(d) + 1);  // n_calls, out_slot, first_call, pad
        const uint32_t call = call_g - h1.z;
        uint8_t* Rin = R + h0.z * RS;
        // the operand progressions four at a time (one 16-byte load for four bases, one for four strides)
        static_assert(kMaxGroupInputs == 8, "two halves of four");
        auto gather4 = [&](uint32_t k0) {
            const uint4 bq = __ldg(reinterpret_cast<const uint4*>(d->in_base + k0));
            const uint4 sq = __ldg(reinterpret_cast<const uint4*>(d->in_stride + k0));
            const uint32_t bs[4] = {bq.x, bq.y, bq.z, bq.w}, ss[4] = {sq.x, sq.y, sq.z, sq.w};
#pragma unroll
            for (uint32_t k = 0; k < 4; k++) {
                if (k0 + k < h0.w) {
                    const uint32_t slot = ss[k] == kTableStride ? __ldg(tables + bs[k] + call) : bs[k] + ss[k] * call;
                    *reinterpret_cast<V*>(Rin + (k0 + k) * RS) = vstore[((size_t)slot << log2_vecs) + vw];
                }
            }
        };
        gather4(0);
        if (h0.w > 4) gather4(4);
        const uint4* op = reinterpret_cast<const uint4*>(gops + h0.x);
        uint32_t r[WPT];  // the previous op's result stays in registers: an operand that names it is not re-read (GroupOp::fwd)
#pragma unroll
        for (int k = 0; k < WPT; k++) r[k] = 0;
#pragma unroll 2
        for (uint32_t i = 0; i < h0.y; i++) {
            // dst_off, a_off, b_off (in units of one register row: x WPT here), fwd  |  m_and, m_xor, m_a, m_c
            const uint4 o = PARAM_OPS ? pops.q[2 * (h0.x + i)] : __ldg(op + 2 * i);
            const uint4 m = PARAM_OPS ? pops.q[2 * (h0.x + i) + 1] : __ldg(op + 2 * i + 1);
            uint32_t a[WPT], b[WPT];
            if (o.w & 1) {
#pragma unroll
                for (int k = 0; k < WPT; k++) a[k] = r[k];
            } else {
                unpack(*reinterpret_cast<const V*>(R + o.y * WPT), a);
            }
            if (o.w & 2) {
#pragma unroll
                for (int k = 0; k < WPT; k++) b[k] = r[k];
            } else {
                unpack(*reinterpret_cast<const V*>(R + o.z * WPT), b);
            }
#pragma unroll
            for (int k = 0; k < WPT; k++) r[k] = (a[k] & b[k] & m.x) ^ ((a[k] ^ b[k]) & m.y) ^ (a[k] & m.z) ^ m.w;
            V v;
            pack(v, r);
            *reinterpret_cast<V*>(R + o.x * WPT) = v;
        }
        const size_t out0 = (size_t)h1.y + (size_t)call * h0.z;
        for (uint32_t k = 0; k < h0.z; k++) vstore[((out0 + k) << log2_vecs) + vw] = *reinterpret_cast<const V*>(R + k * RS);
    }
}

// One call of a prime-field template over a thread's register file R (register r, chunk c at R[(r * NC + c) * T]), shared by
// k_arith_groups and k_arith_chain: the body runs op by op (Montgomery arithmetic of field_ptx.cuh, constants from the
// Montgomery const table), the previous op's result stays in registers (GroupOp::fwd), and an AssertZero tests its
// register in place and reports seq0 + call * A + k.
template <int N, uint32_t FORM, class V>
__device__ __forceinline__ void arith_call(V* R, uint32_t T, const uint4* op, uint32_t n_ops, const uint32_t* __restrict__ consts_mont,
                                           uint32_t seq0, uint32_t call, uint32_t lane, uint32_t* __restrict__ first_fail,
                                           const TileGeom& g, const FieldParams& fp) {
    constexpr int CW = Elem<N>::CW, NC = Elem<N>::NC;
    auto ld_reg = [&](uint32_t* x, uint32_t r) {
#pragma unroll
        for (int c = 0; c < NC; c++) unpack(R[(r * NC + c) * T], x + c * CW);
    };
    auto st_reg = [&](uint32_t r, const uint32_t* x) {
#pragma unroll
        for (int c = 0; c < NC; c++) {
            V v;
            pack(v, x + c * CW);
            R[(r * NC + c) * T] = v;
        }
    };
    uint32_t x[N], y[N], r[N];
#pragma unroll
    for (int k = 0; k < N; k++) r[k] = 0;
    for (uint32_t i = 0; i < n_ops; i++) {
        const uint4 o = __ldg(op + 2 * i);      // dst, a, b registers, fwd
        const uint4 m = __ldg(op + 2 * i + 1);  // kind, const index, assertion ordinal, assertions per call
        if (m.x == AG_CONST) {
#pragma unroll
            for (int k = 0; k < N; k++) r[k] = __ldg(consts_mont + (size_t)m.y * N + k);
            st_reg(o.x, r);
            continue;
        }
        if (o.w & 1) {
#pragma unroll
            for (int k = 0; k < N; k++) x[k] = r[k];
        } else {
            ld_reg(x, o.y);
        }
        if (m.x == AG_ASSERT) {
            const bool fail = !fe_is_zero<N>(x) && lane < g.n_valid;
            report_fail(fail, seq0 + call * m.w + m.z, first_fail, g.batch0 + lane, false);
            continue;
        }
        if (m.x == AG_ADDC || m.x == AG_MULC) {
#pragma unroll
            for (int k = 0; k < N; k++) y[k] = __ldg(consts_mont + (size_t)m.y * N + k);
        } else if (o.w & 2) {
#pragma unroll
            for (int k = 0; k < N; k++) y[k] = r[k];
        } else {
            ld_reg(y, o.z);
        }
        if (m.x == AG_ADD || m.x == AG_ADDC) fe_add<N>(r, x, y, fp.p);
        else fe_mont_mul_form<N, FORM>(r, x, y, fp.p, fp.n0inv);
        st_reg(o.x, r);
    }
}

// Call groups over a prime field: thread <-> (call, witness lane), lane fastest, so for tiles of >= 32 lanes a warp loads
// and stores one coalesced row per 16-byte chunk of the wire store, and for narrower tiles a warp spans calls.  A call's
// inputs are read into a register file in dynamic shared memory, laid out like the wire store with the CTA's threads as
// lanes (chunk c of register r of thread t at ((r * NC + c) * T + t) * CW limbs: a thread's 16-byte chunks are
// conflict-free), arith_call runs the body over it, and only the outputs go back to the wire store (always stored: a group
// output is a level-0 value).  thread -> group as in k_bool_groups.
template <int N, uint32_t FORM>
__global__ void __launch_bounds__(kGroupThreads)
k_arith_groups(const GroupDesc* __restrict__ descs, uint32_t n_groups, uint64_t total_calls, const GroupOp* __restrict__ gops,
               const uint32_t* __restrict__ tables, const uint32_t* __restrict__ hints, uint32_t* __restrict__ store,
               const uint32_t* __restrict__ consts_mont, uint32_t* __restrict__ first_fail, TileGeom g, FieldParams fp) {
    constexpr int CW = Elem<N>::CW, NC = Elem<N>::NC;
    using V = typename Vec<CW>::T;
    extern __shared__ __align__(16) uint8_t s_regs[];
    const uint32_t T = blockDim.x;
    V* R = reinterpret_cast<V*>(s_regs) + threadIdx.x;  // register r, chunk c: R[(r * NC + c) * T]
    auto ld_reg = [&](uint32_t* x, uint32_t r) {
#pragma unroll
        for (int c = 0; c < NC; c++) unpack(R[(r * NC + c) * T], x + c * CW);
    };
    auto st_reg = [&](uint32_t r, const uint32_t* x) {
#pragma unroll
        for (int c = 0; c < NC; c++) {
            V v;
            pack(v, x + c * CW);
            R[(r * NC + c) * T] = v;
        }
    };
    const uint64_t total = total_calls << g.log2_wt;
    const uint32_t wt_mask = (1u << g.log2_wt) - 1;
    for (uint64_t tid = blockIdx.x * (uint64_t)T + threadIdx.x; tid < total; tid += (uint64_t)gridDim.x * T) {
        const uint32_t lane = (uint32_t)tid & wt_mask;
        const uint32_t call_g = (uint32_t)(tid >> g.log2_wt);
        uint32_t gi = __ldg(hints + (call_g >> kGroupHintShift));
        while (gi + 1 < n_groups && call_g >= __ldg(&descs[gi + 1].first_call)) gi++;
        const GroupDesc* d = descs + gi;
        const uint4 h0 = __ldg(reinterpret_cast<const uint4*>(d));      // tmpl_off, n_ops, n_out, n_in
        const uint4 h1 = __ldg(reinterpret_cast<const uint4*>(d) + 1);  // n_calls, out_slot, first_call, seq0
        const uint32_t call = call_g - h1.z;
        uint32_t x[N];
        for (uint32_t k = 0; k < h0.w; k++) {
            const uint32_t base = __ldg(d->in_base + k), st = __ldg(d->in_stride + k);
            const uint32_t slot = st == kTableStride ? __ldg(tables + base + call) : base + st * call;
            load_elem<N>(x, store, slot, lane, g.log2_wt);
            st_reg(h0.z + k, x);
        }
        arith_call<N, FORM>(R, T, reinterpret_cast<const uint4*>(gops + h0.x), h0.y, consts_mont, h1.w, call, lane, first_fail, g, fp);
        const uint32_t out0 = h1.y + call * h0.z;
        for (uint32_t k = 0; k < h0.z; k++) {
            ld_reg(x, k);
            store_elem<N>(store, out0 + k, lane, g.log2_wt, x);
        }
    }
}

template <int BYTES>
__device__ __forceinline__ void chain_cp_async(void* smem_dst, const void* gmem_src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], %2;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gmem_src), "n"(BYTES)
                 : "memory");
}

// Carried loops over a prime field (Plan::chain_descs): thread <-> (chain, witness lane), lane fastest, and the thread walks
// its chain's calls in order.  A chain takes at least a whole warp (lanes past the tile's idle): chains run different
// templates, and two of them sharing a warp would take turns at every divergent op.  The register file is k_arith_groups' (shared memory, same layout), with two areas past the
// template's registers: each carried input's ring of its last lag values (ring register + c % lag holds the value call c
// reads: a seed for c < lag, then output k of call c - lag, written there when that call ends), and from stage0 (the
// descriptor's first_call) kChainStages staging registers per input, which cp.async fills with the non-carried inputs of the next kChainStages
// calls while the earlier ones run, so the wire store's latency stays off the chain.  Carried values never go through the
// wire store; every call's outputs are stored.
template <int N, uint32_t FORM>
__global__ void __launch_bounds__(kGroupThreads)
k_arith_chain(const GroupDesc* __restrict__ descs, const uint32_t* __restrict__ carry, uint32_t n_chains, const GroupOp* __restrict__ gops,
              const uint32_t* __restrict__ tables, uint32_t* __restrict__ store, const uint32_t* __restrict__ consts_mont,
              uint32_t* __restrict__ first_fail, TileGeom g, FieldParams fp) {
    constexpr int CW = Elem<N>::CW, NC = Elem<N>::NC;
    using V = typename Vec<CW>::T;
    extern __shared__ __align__(16) uint8_t s_regs[];
    const uint32_t T = blockDim.x;
    V* R = reinterpret_cast<V*>(s_regs) + threadIdx.x;
    auto ld_reg = [&](uint32_t* x, uint32_t r) {
#pragma unroll
        for (int c = 0; c < NC; c++) unpack(R[(r * NC + c) * T], x + c * CW);
    };
    auto st_reg = [&](uint32_t r, const uint32_t* x) {
#pragma unroll
        for (int c = 0; c < NC; c++) {
            V v;
            pack(v, x + c * CW);
            R[(r * NC + c) * T] = v;
        }
    };
    const uint32_t log2_span = g.log2_wt > 5 ? g.log2_wt : 5;  // threads per chain
    const uint64_t tid = blockIdx.x * (uint64_t)T + threadIdx.x;
    const uint32_t lane = (uint32_t)tid & ((1u << log2_span) - 1);
    if (tid >= ((uint64_t)n_chains << log2_span) || lane >> g.log2_wt) return;
    const uint32_t gi = (uint32_t)(tid >> log2_span);
    const GroupDesc* d = descs + gi;
    const uint32_t* cw = carry + (size_t)gi * kMaxGroupInputs;
    const uint4 h0 = __ldg(reinterpret_cast<const uint4*>(d));      // tmpl_off, n_ops, n_out, n_in
    const uint4 h1 = __ldg(reinterpret_cast<const uint4*>(d) + 1);  // n_calls, out_slot, stage0, seq0
    const uint32_t stage0 = h1.z;
    const uint4* ops = reinterpret_cast<const uint4*>(gops + h0.x);
    const V* gstore = reinterpret_cast<const V*>(store);
    // call c's non-carried inputs -> its staging registers, asynchronously (one commit group per call, empty past the end)
    auto stage = [&](uint32_t call) {
        for (uint32_t k = 0; k < h0.w && call < h1.x; k++) {
            if (__ldg(cw + k)) continue;
            const uint32_t base = __ldg(d->in_base + k), st = __ldg(d->in_stride + k);
            const uint32_t slot = st == kTableStride ? __ldg(tables + base + call) : base + st * call;
#pragma unroll
            for (int c = 0; c < NC; c++)
                chain_cp_async<CW * 4>(&R[((stage0 + k * kChainStages + call % kChainStages) * NC + c) * T],
                                       gstore + ((((size_t)slot * NC + c) << g.log2_wt) + lane));
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    uint32_t x[N];
    for (uint32_t k = 0; k < h0.w; k++) {  // the seeds -> the rings
        const uint32_t w = __ldg(cw + k);
        if (!w) continue;
        const uint32_t base = __ldg(d->in_base + k), ring = (w >> 16) & 0x7FFF, lag = (w >> 8) & 0xFF;
        for (uint32_t s = 0; s < lag; s++) {
            load_elem<N>(x, store, __ldg(tables + base + s), lane, g.log2_wt);
            st_reg(ring + s, x);
        }
    }
    for (uint32_t s = 0; s < kChainStages; s++) stage(s);
    for (uint32_t call = 0; call < h1.x; call++) {
        asm volatile("cp.async.wait_group %0;" ::"n"(kChainStages - 1) : "memory");  // this call's group has landed
        for (uint32_t k = 0; k < h0.w; k++) {
            const uint32_t w = __ldg(cw + k);
            ld_reg(x, w ? ((w >> 16) & 0x7FFF) + call % ((w >> 8) & 0xFF) : stage0 + k * kChainStages + call % kChainStages);
            st_reg(h0.z + k, x);
        }
        stage(call + kChainStages);
        arith_call<N, FORM>(R, T, ops, h0.y, consts_mont, h1.w, call, lane, first_fail, g, fp);
        for (uint32_t k = 0; k < h0.w; k++) {  // output k of this call is what call + lag reads
            const uint32_t w = __ldg(cw + k);
            if (!w) continue;
            ld_reg(x, w & 0xFF);
            st_reg(((w >> 16) & 0x7FFF) + call % ((w >> 8) & 0xFF), x);
        }
        const uint32_t out0 = h1.y + call * h0.z;
        for (uint32_t k = 0; k < h0.z; k++) {
            ld_reg(x, k);
            store_elem<N>(store, out0 + k, lane, g.log2_wt, x);
        }
    }
}

__global__ void k_bool_read_values(const uint32_t* __restrict__ slots, uint32_t n, const uint32_t* __restrict__ store, uint32_t lane,
                                   uint32_t log2_wt, uint32_t* __restrict__ out) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t word = store[((size_t)slots[i] << (log2_wt - 5)) + (lane >> 5)];
    out[i] = (word >> (lane & 31)) & 1;
}

// ---------------------------------------------------------------------------------------------
// capture list (zkb_capture_values): after a tile's last wavefront, the chosen values of every lane -> a witness-major buffer,
// in the bytes zkb_read_values returns.  A CTA holds 32 lanes x VB values (blockDim = 32 x VB): the reads are coalesced over
// lanes (the store is witness-minor), the tile is transposed through shared memory, and the writes are coalesced over values
// (witness j's VB values are VB * E consecutive bytes of the output).
// ---------------------------------------------------------------------------------------------
constexpr uint32_t kCaptureLanes = 32;

template <int N>  // N = 0: p = 2, one bit per lane
__device__ __forceinline__ void capture_tile(const CaptureDesc* __restrict__ descs, uint32_t n, const uint32_t* __restrict__ store,
                                             const InputDesc& in, const uint8_t* __restrict__ raw_consts, uint32_t raw_stride,
                                             const TileGeom& g, uint32_t ew, uint32_t* __restrict__ out, const FieldParams& fp) {
    extern __shared__ uint32_t cap_sm[];
    const uint32_t vb = blockDim.y;
    const uint32_t row = vb * ew + 1;  // words per lane; the odd pitch puts the lanes of a warp in different banks
    const uint32_t l = threadIdx.x, v = threadIdx.y;
    const uint32_t i0 = blockIdx.x * vb, i = i0 + v;
    const uint32_t nv = min(vb, n - i0);
    const uint32_t n_lane_blocks = (g.n_valid + kCaptureLanes - 1) / kCaptureLanes;
    CaptureDesc d{0, 0, 0, 0};
    if (i < n) d = descs[i];
    for (uint32_t lb = blockIdx.y; lb < n_lane_blocks; lb += gridDim.y) {
        const uint32_t j = lb * kCaptureLanes + l;  // lane of the tile
        uint32_t* dst = cap_sm + l * row + v * ew;
        if (i < n && j < g.n_valid) {
            uint32_t w = 0;  // words written
            if (d.kind == CAP_STORE) {
                if constexpr (N == 0) {
                    dst[0] = (store[((size_t)d.slot << (g.log2_wt - 5)) + (j >> 5)] >> (j & 31)) & 1;
                    w = 1;
                } else {
                    uint32_t a[N], one[N], r[N];
                    load_elem<N>(a, store, d.slot, j, g.log2_wt);
#pragma unroll
                    for (int k = 0; k < N; k++) one[k] = (k == 0);
                    fe_mont_mul<N>(r, a, one, fp.p, fp.n0inv);  // leave Montgomery form, as k_read_values does
#pragma unroll
                    for (int k = 0; k < N; k++) dst[k] = r[k];
                    w = N;
                }
            } else {  // raw bytes: an input value as the reference holds it, or a constant >= p
                const uint8_t* src;
                uint32_t len;
                if (d.kind == CAP_RAW_CONST) {
                    src = raw_consts + (size_t)d.opb * raw_stride;
                    len = raw_stride;
                } else {
                    const uint64_t widx = g.batch0 + j;
                    src = (d.kind == CAP_INSTANCE ? in.inst + widx * in.inst_set_stride : in.wit + widx * in.wit_set_stride) +
                          (uint64_t)d.opb * in.stride;
                    len = in.stride;
                }
                for (; 4 * w < len; w++) {
                    uint32_t x = 0;
                    for (uint32_t b = 0; b < 4 && 4 * w + b < len; b++) x |= (uint32_t)src[4 * w + b] << (8 * b);
                    dst[w] = x;
                }
            }
            for (; w < ew; w++) dst[w] = 0;
        }
        __syncthreads();
        const uint32_t nl = min(kCaptureLanes, g.n_valid - lb * kCaptureLanes);
        const uint32_t per_lane = nv * ew;
        for (uint32_t q = v * kCaptureLanes + l; q < nl * per_lane; q += vb * kCaptureLanes) {
            const uint32_t ll = q / per_lane, r = q - ll * per_lane;
            out[((size_t)(g.batch0 + lb * kCaptureLanes + ll) * n + i0) * ew + r] = cap_sm[ll * row + r];
        }
        __syncthreads();
    }
}

template <int N>
__global__ void __launch_bounds__(256)
k_capture(const CaptureDesc* __restrict__ descs, uint32_t n, const uint32_t* __restrict__ store, InputDesc in,
          const uint8_t* __restrict__ raw_consts, uint32_t raw_stride, TileGeom g, uint32_t ew, uint32_t* __restrict__ out, FieldParams fp) {
    capture_tile<N>(descs, n, store, in, raw_consts, raw_stride, g, ew, out, fp);
}

__global__ void __launch_bounds__(256)
k_bool_capture(const CaptureDesc* __restrict__ descs, uint32_t n, const uint32_t* __restrict__ store, InputDesc in,
               const uint8_t* __restrict__ raw_consts, uint32_t raw_stride, TileGeom g, uint32_t ew, uint32_t* __restrict__ out, FieldParams fp) {
    capture_tile<0>(descs, n, store, in, raw_consts, raw_stride, g, ew, out, fp);
}

// a captured value that no gate reads (F_SINK) must be stored on every tile: clear the flag of the op producing it
__global__ void k_unsink(GateOp* ops, uint64_t n_ops, const uint32_t* __restrict__ slot_bits, uint32_t* found, uint32_t cap, uint32_t* n_found) {
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n_ops; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t m = ops[i].meta;
        if (!(m & F_SINK)) continue;
        const uint32_t s = ops[i].out;
        if (!((slot_bits[s >> 5] >> (s & 31)) & 1)) continue;
        ops[i].meta = m & ~F_SINK;
        const uint32_t k = atomicAdd(n_found, 1u);
        if (k < cap) found[k] = (uint32_t)i;
    }
}

__global__ void k_set_sink(GateOp* ops, const uint32_t* __restrict__ idx, uint32_t n, uint32_t set) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    GateOp& op = ops[idx[i]];
    op.meta = set ? (op.meta | F_SINK) : (op.meta & ~F_SINK);
}

__global__ void k_fill_u32(uint32_t* p, uint32_t v, uint64_t n) {
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) p[i] = v;
}

// ---------------------------------------------------------------------------------------------
// launch wrappers
// ---------------------------------------------------------------------------------------------
// experiment knobs (environment, read once): ZKB_LEVEL_PIPE=0/1 selects the software-pipelined hot kernel,
// ZKB_GRID_PER_SM the number of CTAs per SM of the persistent-style grids
static bool level_pipe_enabled() {
    static int v = -1;
    if (v < 0) {
        const char* e = getenv("ZKB_LEVEL_PIPE");
        v = e ? (atoi(e) != 0) : 1;
    }
    return v != 0;
}
// full 256-lane tiles of an 8-limb field go through k_level_tma; ZKB_LEVEL_TMA=0 keeps them on k_level_pipe (read at every
// launch so that one process can compare the two)
static bool level_tma_enabled() {
    const char* e = getenv("ZKB_LEVEL_TMA");
    return e ? atoi(e) != 0 : true;
}
static int grid_per_sm(int dflt) {
    static int v = -1;
    if (v < 0) {
        const char* e = getenv("ZKB_GRID_PER_SM");
        v = e ? atoi(e) : 0;
    }
    return v > 0 ? v : dflt;
}

static inline unsigned grid_for(uint64_t total, int sm_count, int per_sm) {
    uint64_t blocks = (total + 255) / 256;
    uint64_t cap = (uint64_t)sm_count * per_sm;
    if (blocks > cap) blocks = cap;
    if (blocks == 0) blocks = 1;
    return (unsigned)blocks;
}

#define ZKB_DISPATCH_N(nlimb, CALL)         \
    switch (nlimb) {                        \
        case 1: { constexpr int N = 1; CALL; } break; \
        case 2: { constexpr int N = 2; CALL; } break; \
        case 4: { constexpr int N = 4; CALL; } break; \
        default: { constexpr int N = 8; CALL; } break; \
    }

void launch_to_mont(int nlimb, uint32_t* consts, uint32_t n, const FieldParams& fp, cudaStream_t s) {
    if (n == 0) return;
    ZKB_DISPATCH_N(nlimb, (k_to_mont<N><<<(n + 127) / 128, 128, 0, s>>>(consts, n, fp)));
}

void launch_load_inputs(int nlimb, const InputLoad* loads, uint32_t n_loads, uint32_t* store, const uint32_t* consts_mont,
                        InputDesc in, TileGeom g, uint32_t* unreduced_count, uint8_t* rawflag, const uint8_t* const_flags,
                        const FieldParams& fp, int sm_count, cudaStream_t s) {
    if (n_loads == 0) return;
    unsigned grid = grid_for((uint64_t)n_loads << g.log2_wt, sm_count, 256);
    ZKB_DISPATCH_N(nlimb, (k_load_inputs<N><<<grid, 256, 0, s>>>(loads, n_loads, store, consts_mont, in, g, unreduced_count, rawflag,
                                                                 const_flags, fp)));
}

void launch_level(int nlimb, const GateOp* ops, const uint32_t* aseq, uint64_t n_ops, uint32_t* store,
                  const uint32_t* consts_mont, uint32_t* first_fail, const RawCtx& rc, TileGeom g, const FieldParams& fp,
                  int sm_count, bool rare, cudaStream_t s) {
    if (n_ops == 0) return;
    // grid: a whole number of CTAs per SM (multiple of the SM count), grid-stride inside.  Measured on B200
    // (scripts/ab_level.sh, C3): 8 CTAs/SM (exactly resident, static partition) 87 % of the HBM roofline,
    // 64/SM 92.7 %, 256/SM 92.9 % — many more CTAs than are resident lets the hardware scheduler even out
    // the DRAM-locality differences between SMs, while each thread still pipelines several gates.
    unsigned grid = grid_for(n_ops << g.log2_wt, sm_count, grid_per_sm(256));
    if (!rare) {
        if (level_pipe_enabled()) {
            // narrow fields: 4 (one limb) or 2 (two limbs) witness lanes per thread when the tile still gives every warp
            // 32 packed lanes of one gate (ZKB_LEVEL_LPT=1 switches the packing off)
            static const bool pack = getenv("ZKB_LEVEL_LPT") == nullptr || atoi(getenv("ZKB_LEVEL_LPT")) != 1;
            if (pack && nlimb == 2 && g.log2_wt >= 6) {
                grid = grid_for(n_ops << (g.log2_wt - 1), sm_count, grid_per_sm(256));
                k_level_pipe<2, 2><<<grid, 256, 0, s>>>(ops, aseq, n_ops, store, consts_mont, first_fail, g, fp);
            } else if (pack && nlimb == 1 && g.log2_wt >= 7) {
                grid = grid_for(n_ops << (g.log2_wt - 2), sm_count, grid_per_sm(256));
                k_level_pipe<1, 4><<<grid, 256, 0, s>>>(ops, aseq, n_ops, store, consts_mont, first_fail, g, fp);
            } else if (nlimb == 8 && g.log2_wt >= 8 && level_tma_enabled()) {
                static int tma_per_sm = 0;
                static std::atomic<uint64_t> tma_attr_seen{0};
                constexpr size_t smem = kTmaSmemBytes;
                if (first_on_device(tma_attr_seen)) {
                    cudaFuncSetAttribute(k_level_tma<8, kMulFormGeneric>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
                    cudaFuncSetAttribute(k_level_tma<8, kMulFormLow64>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
                }
                if (!tma_per_sm) {
                    const char* e = getenv("ZKB_TMA_GRID_PER_SM");
                    tma_per_sm = e ? std::max(1, atoi(e)) : 128;
                }
                grid = grid_for(n_ops << g.log2_wt, sm_count, tma_per_sm);
                if (fp.mul_form == kMulFormLow64)
                    k_level_tma<8, kMulFormLow64><<<grid, 256, smem, s>>>(ops, aseq, n_ops, store, consts_mont, first_fail, g, fp);
                else
                    k_level_tma<8, kMulFormGeneric><<<grid, 256, smem, s>>>(ops, aseq, n_ops, store, consts_mont, first_fail, g, fp);
            } else if (nlimb == 8 && fp.mul_form == kMulFormLow64) {
                k_level_pipe<8, 1, kMulFormLow64><<<grid, 256, 0, s>>>(ops, aseq, n_ops, store, consts_mont, first_fail, g, fp);
            } else {
                ZKB_DISPATCH_N(nlimb, (k_level_pipe<N, 1><<<grid, 256, 0, s>>>(ops, aseq, n_ops, store, consts_mont, first_fail, g, fp)));
            }
        } else {
            ZKB_DISPATCH_N(nlimb, (k_level<N, false><<<grid, 256, 0, s>>>(ops, aseq, n_ops, store, consts_mont, first_fail, rc, g, fp)));
        }
    } else {
        ZKB_DISPATCH_N(nlimb, (k_level<N, true><<<grid, 256, 0, s>>>(ops, aseq, n_ops, store, consts_mont, first_fail, rc, g, fp)));
    }
}

template <int N>
static cudaError_t launch_coop_n(const GateOp* ops, const uint32_t* aseq, const uint64_t* level_off, uint32_t n_levels, uint32_t* store,
                                 const uint32_t* consts_mont, uint32_t* first_fail, RawCtx rc, TileGeom g, FieldParams fp,
                                 int sm_count, uint64_t max_level_items, uint32_t* barrier_ctr, uint32_t* barrier_epoch, cudaStream_t s) {
    // cooperative_groups' grid.sync() measured faster than the counter barrier (1.19 vs 1.81 us at 444 CTAs, 1.18 vs 1.25 at
    // 148; C2 4.40 vs 4.74 us per level: profiles/r02h_ab_c2.log), so it stays the default; ZKB_COUNTER_BARRIER=1 for the A/B
    static const bool counter_barrier = getenv("ZKB_COUNTER_BARRIER") != nullptr;
    if (!counter_barrier) barrier_ctr = nullptr;
    uint32_t barrier_base = *barrier_epoch;
    void* args[] = {(void*)&ops, (void*)&aseq, (void*)&level_off, (void*)&n_levels, (void*)&store, (void*)&consts_mont,
                    (void*)&first_fail, (void*)&rc, (void*)&g, (void*)&fp, (void*)&barrier_ctr, (void*)&barrier_base};
    // a wavefront that fits one cluster of 8 x 512 threads (two items per thread at most): cluster barrier
    static const bool no_cluster = getenv("ZKB_NO_CLUSTER") != nullptr;
    static bool cluster_ok = true;
    if (!no_cluster && cluster_ok && max_level_items <= 8 * 512 * 2) {
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(8);
        cfg.blockDim = dim3(512);
        cfg.stream = s;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = 8;
        attr[0].val.clusterDim.y = 1;
        attr[0].val.clusterDim.z = 1;
        cfg.attrs = attr;
        cfg.numAttrs = 1;
        cudaError_t ec = cudaLaunchKernelExC(&cfg, (const void*)k_levels_coop<N, true>, args);
        if (ec == cudaSuccess) return ec;
        cudaGetLastError();
        cluster_ok = false;  // not launchable as a cluster here: grid barrier below
    }
    int per_sm = 0;
    cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_levels_coop<N, false>, 256, 0);
    if (e != cudaSuccess) return e;
    if (per_sm < 1) return cudaErrorLaunchOutOfResources;
    // the grid barrier costs more the more CTAs take part: use only as many CTAs (a multiple of the SM count)
    // as the widest level can occupy
    uint64_t want = (max_level_items + 255) / 256;
    uint64_t blocks = ((want + sm_count - 1) / sm_count) * sm_count;
    if (blocks < (uint64_t)sm_count) blocks = sm_count;
    if (blocks > (uint64_t)sm_count * per_sm) blocks = (uint64_t)sm_count * per_sm;
    if (const char* e = getenv("ZKB_COOP_BLOCKS")) blocks = (uint64_t)atoi(e);
    e = cudaLaunchCooperativeKernel((void*)k_levels_coop<N, false>, dim3((unsigned)blocks), dim3(256), args, 0, s);
    if (e == cudaSuccess && barrier_ctr && n_levels > 1) *barrier_epoch += (uint32_t)blocks * (n_levels - 1);  // arrivals this launch adds
    return e;
}

// barrier micro-benchmark: n barriers and nothing else (zkb_debug_barrier_cost)
template <int KIND>
__global__ void __launch_bounds__(KIND == 2 ? 512 : 256) k_barrier_only(uint32_t n, uint32_t* ctr, uint32_t base, uint32_t* sink) {
    uint32_t acc = 0;
    for (uint32_t i = 0; i < n; i++) {
        if (KIND == 0) cg::this_grid().sync();
        else if (KIND == 1) grid_barrier(ctr, base + gridDim.x * (i + 1));
        else cg::this_cluster().sync();
        acc += i;
    }
    if (acc == 0xFFFFFFFFu) *sink = acc;
}

cudaError_t measure_barrier_cost(int kind, unsigned blocks, unsigned n_barriers, uint32_t* barrier_ctr, uint32_t* barrier_epoch,
                                 cudaStream_t s, cudaEvent_t ev0, cudaEvent_t ev1, float* us_per_barrier) {
    uint32_t base = *barrier_epoch;
    uint32_t* sink = barrier_ctr;  // never written
    float best = 1e30f;
    for (int rep = 0; rep < 4; rep++) {
        // the launch itself is timed too: subtract an n = 0 launch of the same shape
        float ms[2] = {0, 0};
        for (int pass = 0; pass < 2; pass++) {
            uint32_t n = pass == 0 ? 0u : n_barriers;
            base = *barrier_epoch;
            void* args[] = {(void*)&n, (void*)&barrier_ctr, (void*)&base, (void*)&sink};
            cudaEventRecord(ev0, s);
            cudaError_t e;
            if (kind == 2) {
                cudaLaunchConfig_t cfg = {};
                cfg.gridDim = dim3(8);
                cfg.blockDim = dim3(512);
                cfg.stream = s;
                cudaLaunchAttribute attr[1];
                attr[0].id = cudaLaunchAttributeClusterDimension;
                attr[0].val.clusterDim.x = 8;
                attr[0].val.clusterDim.y = 1;
                attr[0].val.clusterDim.z = 1;
                cfg.attrs = attr;
                cfg.numAttrs = 1;
                e = cudaLaunchKernelExC(&cfg, (const void*)k_barrier_only<2>, args);
            } else if (kind == 1) {
                e = cudaLaunchCooperativeKernel((void*)k_barrier_only<1>, dim3(blocks), dim3(256), args, 0, s);
                if (e == cudaSuccess) *barrier_epoch += blocks * n;
            } else {
                e = cudaLaunchCooperativeKernel((void*)k_barrier_only<0>, dim3(blocks), dim3(256), args, 0, s);
            }
            if (e != cudaSuccess) return e;
            cudaEventRecord(ev1, s);
            e = cudaStreamSynchronize(s);
            if (e != cudaSuccess) return e;
            cudaEventElapsedTime(&ms[pass], ev0, ev1);
        }
        if (rep > 0) best = std::min(best, ms[1] - ms[0]);
    }
    *us_per_barrier = best * 1e3f / (float)n_barriers;
    return cudaSuccess;
}

cudaError_t launch_levels_coop(int nlimb, const GateOp* ops, const uint32_t* aseq, const uint64_t* level_off, uint32_t n_levels,
                               uint32_t* store, const uint32_t* consts_mont, uint32_t* first_fail, const RawCtx& rc, TileGeom g,
                               const FieldParams& fp, int sm_count, uint64_t max_level_items, uint32_t* barrier_ctr,
                               uint32_t* barrier_epoch, cudaStream_t s) {
    cudaError_t e = cudaSuccess;
    ZKB_DISPATCH_N(nlimb, (e = launch_coop_n<N>(ops, aseq, level_off, n_levels, store, consts_mont, first_fail, rc, g, fp, sm_count,
                                                max_level_items, barrier_ctr, barrier_epoch, s)));
    return e;
}

// the dataflow launch (k_levels_flow): one witness, 1- or 2-limb field, plan without slot re-use.  `fill_from` .. `n_slots`
// are the computed slots, marked "not computed yet" first.  cudaErrorNotSupported: not this kernel's case.
template <int N>
static cudaError_t launch_flow_n(const GateOp* ops, const uint32_t* aseq, const uint64_t* level_off, uint32_t n_levels, uint32_t* store,
                                 const uint32_t* consts_mont, uint32_t* first_fail, RawCtx rc, TileGeom g, FieldParams fp, int sm_count,
                                 uint64_t max_level_items, uint32_t fill_from, uint32_t n_slots, cudaStream_t s) {
    int per_sm = 0;
    cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_levels_flow<N>, 256, 0);
    if (e != cudaSuccess) return e;
    if (per_sm < 1) return cudaErrorLaunchOutOfResources;
    uint64_t want = (max_level_items + 255) / 256;
    uint64_t blocks = ((want + sm_count - 1) / sm_count) * sm_count;
    if (blocks < (uint64_t)sm_count) blocks = sm_count;
    if (blocks > (uint64_t)sm_count * per_sm) blocks = (uint64_t)sm_count * per_sm;
    if (const char* eb = getenv("ZKB_FLOW_BLOCKS")) blocks = std::min<uint64_t>((uint64_t)std::max(1, atoi(eb)), (uint64_t)sm_count * per_sm);
    if (n_slots > fill_from) {
        e = cudaMemsetAsync(store + (size_t)fill_from * N, 0xFF, (size_t)(n_slots - fill_from) * N * 4, s);
        if (e != cudaSuccess) return e;
    }
    uint32_t sleep_ns = 0;  // back-off between polls of a marker word (A/B knob)
    if (const char* es = getenv("ZKB_FLOW_SLEEP")) sleep_ns = (uint32_t)atoi(es);
    void* args[] = {(void*)&ops, (void*)&aseq, (void*)&level_off, (void*)&n_levels, (void*)&store, (void*)&consts_mont,
                    (void*)&first_fail, (void*)&rc, (void*)&g, (void*)&fp, (void*)&sleep_ns};
    return cudaLaunchCooperativeKernel((void*)k_levels_flow<N>, dim3((unsigned)blocks), dim3(256), args, 0, s);
}
template <int N>
static cudaError_t launch_flow_wide_n(const GateOp* ops, const uint32_t* aseq, const uint64_t* level_off, uint32_t n_levels, uint32_t* store,
                                      const uint32_t* consts_mont, uint32_t* first_fail, RawCtx rc, TileGeom g, FieldParams fp, int sm_count,
                                      uint64_t max_level_items, uint32_t n_ready, uint32_t* flags, uint32_t epoch, cudaStream_t s) {
    int per_sm = 0;
    cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_levels_flow_wide<N>, 256, 0);
    if (e != cudaSuccess) return e;
    if (per_sm < 1) return cudaErrorLaunchOutOfResources;
    uint64_t want = (max_level_items + 255) / 256;
    uint64_t blocks = ((want + sm_count - 1) / sm_count) * sm_count;
    if (blocks < (uint64_t)sm_count) blocks = sm_count;
    if (blocks > (uint64_t)sm_count * per_sm) blocks = (uint64_t)sm_count * per_sm;
    if (const char* eb = getenv("ZKB_FLOW_BLOCKS")) blocks = std::min<uint64_t>((uint64_t)std::max(1, atoi(eb)), (uint64_t)sm_count * per_sm);
    void* args[] = {(void*)&ops, (void*)&aseq, (void*)&level_off, (void*)&n_levels, (void*)&store, (void*)&consts_mont,
                    (void*)&first_fail, (void*)&rc, (void*)&g, (void*)&fp, (void*)&flags, (void*)&epoch, (void*)&n_ready};
    return cudaLaunchCooperativeKernel((void*)k_levels_flow_wide<N>, dim3((unsigned)blocks), dim3(256), args, 0, s);
}
cudaError_t launch_levels_flow_wide(int nlimb, const GateOp* ops, const uint32_t* aseq, const uint64_t* level_off, uint32_t n_levels,
                                    uint32_t* store, const uint32_t* consts_mont, uint32_t* first_fail, const RawCtx& rc, TileGeom g,
                                    const FieldParams& fp, int sm_count, uint64_t max_level_items, uint32_t n_ready, uint32_t* flags,
                                    uint32_t epoch, cudaStream_t s) {
    if (g.log2_wt != 0) return cudaErrorNotSupported;
    if (nlimb == 4) return launch_flow_wide_n<4>(ops, aseq, level_off, n_levels, store, consts_mont, first_fail, rc, g, fp, sm_count, max_level_items, n_ready, flags, epoch, s);
    if (nlimb == 8) return launch_flow_wide_n<8>(ops, aseq, level_off, n_levels, store, consts_mont, first_fail, rc, g, fp, sm_count, max_level_items, n_ready, flags, epoch, s);
    return cudaErrorNotSupported;
}

cudaError_t launch_levels_flow(int nlimb, const GateOp* ops, const uint32_t* aseq, const uint64_t* level_off, uint32_t n_levels,
                               uint32_t* store, const uint32_t* consts_mont, uint32_t* first_fail, const RawCtx& rc, TileGeom g,
                               const FieldParams& fp, int sm_count, uint64_t max_level_items, uint32_t fill_from, uint32_t n_slots,
                               cudaStream_t s) {
    if (g.log2_wt != 0) return cudaErrorNotSupported;
    if (nlimb == 1) return launch_flow_n<1>(ops, aseq, level_off, n_levels, store, consts_mont, first_fail, rc, g, fp, sm_count, max_level_items, fill_from, n_slots, s);
    if (nlimb == 2) return launch_flow_n<2>(ops, aseq, level_off, n_levels, store, consts_mont, first_fail, rc, g, fp, sm_count, max_level_items, fill_from, n_slots, s);
    return cudaErrorNotSupported;
}

void launch_read_values(int nlimb, const uint32_t* slots, uint32_t n, const uint32_t* store, uint32_t lane, uint32_t log2_wt,
                        uint32_t* out, const FieldParams& fp, cudaStream_t s) {
    if (n == 0) return;
    ZKB_DISPATCH_N(nlimb, (k_read_values<N><<<(n + 127) / 128, 128, 0, s>>>(slots, n, store, lane, log2_wt, out, fp)));
}

void launch_bool_load_inputs(const InputLoad* loads, uint32_t n_loads, uint32_t* store, const uint32_t* const_bits, InputDesc in,
                             TileGeom g, uint32_t* unreduced_count, uint8_t* rawflag, const uint8_t* const_flags, int sm_count,
                             cudaStream_t s) {
    if (n_loads == 0) return;
    unsigned grid = grid_for((uint64_t)n_loads << g.log2_wt, sm_count, 256);
    k_bool_load_inputs<<<grid, 256, 0, s>>>(loads, n_loads, store, const_bits, in, g, unreduced_count, rawflag, const_flags);
}

void launch_bool_level(const GateOp* ops, const uint32_t* aseq, uint64_t n_ops, uint32_t* store, const uint32_t* const_bits,
                       uint32_t* first_fail, const uint8_t* rawflag, TileGeom g, int sm_count, cudaStream_t s) {
    if (n_ops == 0) return;
    if (g.log2_wt >= 7) {  // >= 128 witnesses: four words per thread
        unsigned grid = grid_for(n_ops << (g.log2_wt - 7), sm_count, grid_per_sm(256));
        k_bool_level<4><<<grid, 256, 0, s>>>(ops, aseq, n_ops, store, const_bits, first_fail, rawflag, g);
    } else {
        unsigned grid = grid_for(n_ops << (g.log2_wt - 5), sm_count, grid_per_sm(256));
        k_bool_level<1><<<grid, 256, 0, s>>>(ops, aseq, n_ops, store, const_bits, first_fail, rawflag, g);
    }
}

void launch_bool_levels_cta(const GateOp* ops, const uint32_t* aseq, const uint64_t* level_off, uint32_t n_levels, uint32_t* store,
                            const uint32_t* const_bits, uint32_t* first_fail, const uint8_t* rawflag, TileGeom g, cudaStream_t s) {
    if (n_levels == 0) return;
    if (g.log2_wt >= 7) k_bool_levels_cta<4><<<1, 256, 0, s>>>(ops, aseq, level_off, n_levels, store, const_bits, first_fail, rawflag, g);
    else k_bool_levels_cta<1><<<1, 256, 0, s>>>(ops, aseq, level_off, n_levels, store, const_bits, first_fail, rawflag, g);
}

void launch_bool_groups(const GroupDesc* descs, uint32_t n_groups, uint64_t total_calls, const GroupOp* gops, const uint32_t* tables,
                        const uint32_t* hints, uint32_t* store, TileGeom g, uint32_t n_regs, int sm_count, cudaStream_t s,
                        const GroupOp* host_ops, uint32_t n_host_ops) {
    if (n_groups == 0 || total_calls == 0) return;
    static std::atomic<uint64_t> attr_seen{0};
    if (first_on_device(attr_seen)) {  // up to kMaxTemplateRegs x 256 threads x 16 bytes
        cudaFuncSetAttribute(k_bool_groups<1, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(kMaxTemplateRegs * kGroupThreads * 4));
        cudaFuncSetAttribute(k_bool_groups<4, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(kMaxTemplateRegs * kGroupThreads * 16));
        cudaFuncSetAttribute(k_bool_groups<1, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(kMaxTemplateRegs * kGroupThreads * 4));
        cudaFuncSetAttribute(k_bool_groups<4, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(kMaxTemplateRegs * kGroupThreads * 16));
    }
    const uint32_t log2_words = g.log2_wt - 5;
    const bool wide = log2_words >= 2;
    const size_t smem = (size_t)n_regs * kGroupThreads * (wide ? 16 : 4);
    const uint64_t total = total_calls << (wide ? log2_words - 2 : log2_words);
    const uint64_t tiles = (total + kGroupThreads - 1) / kGroupThreads;
    const unsigned grid = (unsigned)std::min<uint64_t>(tiles, (uint64_t)sm_count * 64);
    static GroupOpsParam none{};
    const bool in_params = host_ops != nullptr && n_host_ops <= kGroupParamOps && getenv("ZKB_GROUP_OPS_GLOBAL") == nullptr;
    if (in_params) {
        GroupOpsParam pp;
        memcpy(pp.q, host_ops, (size_t)n_host_ops * sizeof(GroupOp));
        if (wide) k_bool_groups<4, true><<<grid, kGroupThreads, smem, s>>>(descs, n_groups, total_calls, gops, tables, hints, store, log2_words, pp);
        else k_bool_groups<1, true><<<grid, kGroupThreads, smem, s>>>(descs, n_groups, total_calls, gops, tables, hints, store, log2_words, pp);
    } else {
        if (wide) k_bool_groups<4, false><<<grid, kGroupThreads, smem, s>>>(descs, n_groups, total_calls, gops, tables, hints, store, log2_words, none);
        else k_bool_groups<1, false><<<grid, kGroupThreads, smem, s>>>(descs, n_groups, total_calls, gops, tables, hints, store, log2_words, none);
    }
}

// CTA size: the largest power of two <= 256 threads whose register file (n_regs x 4N bytes a thread) leaves room for two
// CTAs per SM
static constexpr size_t kArithGroupSmemPerCta = 112 * 1024;
uint32_t arith_group_threads(int nlimb, uint32_t n_regs) {
    uint32_t t = kGroupThreads;
    while (t > 32 && (size_t)n_regs * nlimb * 4 * t > kArithGroupSmemPerCta) t >>= 1;
    return t;
}
template <int N, uint32_t FORM>
static void launch_arith_groups_n(const GroupDesc* descs, uint32_t n_groups, uint64_t total_calls, const GroupOp* gops, const uint32_t* tables,
                                  const uint32_t* hints, uint32_t* store, const uint32_t* consts_mont, uint32_t* first_fail, TileGeom g,
                                  const FieldParams& fp, uint32_t n_regs, int sm_count, cudaStream_t s) {
    static std::atomic<uint64_t> attr_seen{0};
    if (first_on_device(attr_seen)) cudaFuncSetAttribute(k_arith_groups<N, FORM>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kArithGroupSmemPerCta);
    const uint32_t T = arith_group_threads(N, n_regs);
    const size_t smem = (size_t)std::max<uint32_t>(n_regs, 1) * N * 4 * T;
    const uint64_t blocks = ((total_calls << g.log2_wt) + T - 1) / T;
    const unsigned grid = (unsigned)std::min<uint64_t>(blocks, (uint64_t)sm_count * (2048 / T));
    k_arith_groups<N, FORM><<<grid, T, smem, s>>>(descs, n_groups, total_calls, gops, tables, hints, store, consts_mont, first_fail, g, fp);
}
void launch_arith_groups(int nlimb, const GroupDesc* descs, uint32_t n_groups, uint64_t total_calls, const GroupOp* gops, const uint32_t* tables,
                         const uint32_t* hints, uint32_t* store, const uint32_t* consts_mont, uint32_t* first_fail, TileGeom g,
                         const FieldParams& fp, uint32_t n_regs, int sm_count, cudaStream_t s) {
    if (n_groups == 0 || total_calls == 0) return;
    if (nlimb == 8 && fp.mul_form == kMulFormLow64)
        launch_arith_groups_n<8, kMulFormLow64>(descs, n_groups, total_calls, gops, tables, hints, store, consts_mont, first_fail, g, fp, n_regs,
                                                sm_count, s);
    else
        ZKB_DISPATCH_N(nlimb, (launch_arith_groups_n<N, kMulFormGeneric>(descs, n_groups, total_calls, gops, tables, hints, store, consts_mont,
                                                                         first_fail, g, fp, n_regs, sm_count, s)));
}

// CTA size: as k_arith_groups' (two CTAs per SM), and smaller while that leaves SMs idle: each thread is a serial walk,
// latency-bound, so the threads are spread over the SMs rather than stacked on a few
template <int N, uint32_t FORM>
static void launch_arith_chain_n(const GroupDesc* descs, const uint32_t* carry, uint32_t n_chains, const GroupOp* gops, const uint32_t* tables,
                                 uint32_t* store, const uint32_t* consts_mont, uint32_t* first_fail, TileGeom g, const FieldParams& fp,
                                 uint32_t n_regs, int sm_count, cudaStream_t s) {
    static std::atomic<uint64_t> attr_seen{0};
    if (first_on_device(attr_seen)) cudaFuncSetAttribute(k_arith_chain<N, FORM>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kArithGroupSmemPerCta);
    const uint64_t threads = (uint64_t)n_chains << (g.log2_wt > 5 ? g.log2_wt : 5);  // a warp at least per chain
    uint32_t T = arith_group_threads(N, n_regs);
    while (T > 32 && (threads + T - 1) / T < (uint64_t)sm_count) T >>= 1;
    const size_t smem = (size_t)n_regs * N * 4 * T;
    k_arith_chain<N, FORM><<<(unsigned)((threads + T - 1) / T), T, smem, s>>>(descs, carry, n_chains, gops, tables, store, consts_mont, first_fail,
                                                                            g, fp);
}
void launch_arith_chain(int nlimb, const GroupDesc* descs, const uint32_t* carry, uint32_t n_chains, const GroupOp* gops, const uint32_t* tables,
                        uint32_t* store, const uint32_t* consts_mont, uint32_t* first_fail, TileGeom g, const FieldParams& fp, uint32_t n_regs,
                        int sm_count, cudaStream_t s) {
    if (n_chains == 0) return;
    if (nlimb == 8 && fp.mul_form == kMulFormLow64)
        launch_arith_chain_n<8, kMulFormLow64>(descs, carry, n_chains, gops, tables, store, consts_mont, first_fail, g, fp, n_regs, sm_count, s);
    else
        ZKB_DISPATCH_N(nlimb, (launch_arith_chain_n<N, kMulFormGeneric>(descs, carry, n_chains, gops, tables, store, consts_mont, first_fail, g,
                                                                        fp, n_regs, sm_count, s)));
}

void launch_bool_read_values(const uint32_t* slots, uint32_t n, const uint32_t* store, uint32_t lane, uint32_t log2_wt,
                             uint32_t* out, cudaStream_t s) {
    if (n == 0) return;
    k_bool_read_values<<<(n + 127) / 128, 128, 0, s>>>(slots, n, store, lane, log2_wt, out);
}

template <class K>
static cudaError_t launch_capture_k(K kernel, const CaptureDesc* descs, uint32_t n, const uint32_t* store, const InputDesc& in,
                                   const uint8_t* raw_consts, uint32_t raw_stride, const TileGeom& g, uint32_t ew, uint8_t* out,
                                   const FieldParams& fp, cudaStream_t s) {
    // 8 values a CTA (256 threads) while the transpose buffer fits the default 48 KB, fewer for wide raw inputs
    auto smem_for = [&](uint32_t vb) { return (size_t)kCaptureLanes * (vb * ew + 1) * 4; };
    uint32_t vb = 8;
    while (vb > 1 && smem_for(vb) > 48 * 1024) vb >>= 1;
    const size_t smem = smem_for(vb);
    if (smem > 48 * 1024) {
        if (smem > 227 * 1024) return cudaErrorInvalidValue;
        cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
    }
    const uint32_t lane_blocks = (g.n_valid + kCaptureLanes - 1) / kCaptureLanes;
    const dim3 grid((n + vb - 1) / vb, std::min<uint32_t>(lane_blocks, 65535));
    kernel<<<grid, dim3(kCaptureLanes, vb), smem, s>>>(descs, n, store, in, raw_consts, raw_stride, g, ew, (uint32_t*)out, fp);
    return cudaPeekAtLastError();
}

cudaError_t launch_capture(int nlimb, const CaptureDesc* descs, uint32_t n, const uint32_t* store, InputDesc in, const uint8_t* raw_consts,
                           uint32_t raw_stride, TileGeom g, uint32_t E, uint8_t* out, const FieldParams& fp, cudaStream_t s) {
    if (n == 0 || g.n_valid == 0) return cudaSuccess;
    cudaError_t e = cudaSuccess;
    if (nlimb == 0) return launch_capture_k(k_bool_capture, descs, n, store, in, raw_consts, raw_stride, g, E / 4, out, fp, s);
    ZKB_DISPATCH_N(nlimb, (e = launch_capture_k(k_capture<N>, descs, n, store, in, raw_consts, raw_stride, g, E / 4, out, fp, s)));
    return e;
}

void launch_unsink(GateOp* ops, uint64_t n_ops, const uint32_t* slot_bits, uint32_t* found, uint32_t cap, uint32_t* n_found, int sm_count,
                   cudaStream_t s) {
    if (n_ops == 0) return;
    k_unsink<<<grid_for(n_ops, sm_count, 8), 256, 0, s>>>(ops, n_ops, slot_bits, found, cap, n_found);
}

void launch_set_sink(GateOp* ops, const uint32_t* idx, uint32_t n, bool set, cudaStream_t s) {
    if (n == 0) return;
    k_set_sink<<<(n + 255) / 256, 256, 0, s>>>(ops, idx, n, set ? 1u : 0u);
}

void launch_fill_u32(uint32_t* p, uint32_t v, uint64_t n, int sm_count, cudaStream_t s) {
    if (n == 0) return;
    k_fill_u32<<<grid_for(n, sm_count, 8), 256, 0, s>>>(p, v, n);
}

}  // namespace zkb
