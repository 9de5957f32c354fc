// R1CS satisfiability as CSR sparse mod-p mat-vecs with a fused Hadamard check
// (section 5 of include/zkb.h).
//
// Reference semantics: `zkif-to-ir` expands every constraint (A_r, B_r, C_r) into
//   per term  Constant(coef) [+ Mul(var, const)],  per LC a chain of Add,
//   Mul(a, b), Mul(-1, c), Add, AssertZero          (rust/src/producers/from_r1cs.rs:71-125)
// and `evaluate` then walks those gates one by one.  Algebraically that is
//   (A_r . z)(B_r . z) - (C_r . z) == 0 (mod p)   for every row r,   z_0 = 1,
// which is what k_r1cs_check computes directly: one thread per (row, witness lane), three CSR
// dot products in Montgomery form and the row test, with the first violated row reported per
// witness (= the first failing AssertZero of the gate expansion, which emits one per row in order).
// No tensor cores: the matrices are ~3 nnz/row sparse, nothing here is a dense contraction.
#include <stdio.h>
#include <string.h>

#include <algorithm>

#include "context.h"
#include "device_util.cuh"

using namespace zkb;

#define CUDA_TRY(c, expr)                                                                              \
    do {                                                                                               \
        cudaError_t e__ = (expr);                                                                      \
        if (e__ != cudaSuccess)                                                                        \
            return (c)->fail(ZKB_E_CUDA, std::string("CUDA error: ") + cudaGetErrorString(e__) + " at " #expr); \
    } while (0)

namespace zkb {

// Device layout of the three matrices: SELL-32-sigma (sliced ELLPACK).  Rows are sorted by their six class counts,
// heaviest first, inside windows of `sigma` consecutive rows (locality of the variables a window touches is kept,
// e.g. the slack variables of neighbouring rows stay in the same L2-resident region) and cut into slices of 32
// sorted rows.  The terms of a row fall in six classes — A, B, C times {coefficient one, general coefficient} — and a
// slice stores K_class groups per class (the slice's largest count of that class); a group is 32 x {col, coef}
// with the row of the slice as the fast index, so
//   - with ONE assignment a warp works on the 32 rows of a slice: every group is one coalesced 256-byte load
//     and all lanes run the same trip counts;
//   - with a batch of assignments a warp works on one row for 32 assignments: the term is a broadcast load and
//     the z gathers are coalesced 512-byte rows.
// Rows shorter than their slice are padded with {0, T_PAD}.
constexpr uint32_t T_PAD = 0xFFFFFFFFu;  // no term
constexpr uint32_t T_ONE = 0xFFFFFFFEu;  // coefficient 1: the multiplication is skipped

// One sliced layout.  Two are kept, built on first use:
//   kind 0 (tiles of < 32 assignments, in particular ONE assignment): six classes, sigma = 262144 rows — the lanes of a
//          warp are different rows, so ones and general terms are separated and sorted on;
//   kind 1 (tiles of >= 32 assignments): a warp is one row, nothing diverges: one class per matrix (ones tagged inside
//          it), sorted by |A_r|, |B_r|, |C_r| only, sigma = 16384 rows so that the window's variables x the tile width
//          stay L2-resident.
struct R1csLayout {
    bool built = false;
    uint64_t n_slices = 0, n_groups = 0;
    uint4* d_slices = nullptr;     // {first group, A ones | A general << 16, B ones | B general << 16, C ones | C general << 16}
    uint2* d_terms = nullptr;      // [group][32] {col, coefficient index | T_ONE | T_PAD}
    uint32_t* d_row_ids = nullptr; // sorted position -> original row (the verdict names the original row)
    // host copies (host-only contexts: zkb_debug_r1cs_layout)
    std::vector<uint4> h_slices;
    std::vector<uint2> h_terms;
    std::vector<uint32_t> h_row_ids;
};

struct R1csDev {
    uint64_t n_rows = 0, n_vars = 0, nnz[3] = {0, 0, 0};
    // the system as loaded, zero coefficients dropped, coefficient one tagged (the layouts are built from this)
    std::vector<uint32_t> h_rp[3], h_col[3], h_tag[3];
    R1csLayout layout[2];
    uint32_t* d_coefs = nullptr;   // Montgomery form, nlimb limbs each
    uint32_t n_coefs = 0;
    uint32_t* d_z = nullptr;       // [var][chunk][lane][CW] Montgomery
    size_t z_bytes = 0;
    uint8_t* d_zraw = nullptr;
    size_t zraw_bytes = 0;
    uint64_t z_set_stride = 0;
    uint32_t stride = 0, n_batch = 0, log2_wt = 0;
    uint32_t* d_first_fail = nullptr;
    size_t first_fail_cap = 0;
    bool uploaded = false;
};

void r1cs_free(zkb_ctx* c) {
    R1csDev* r = c->r1cs;
    if (!r) return;
    for (auto& l : r->layout) {
        cudaFree(l.d_slices);
        cudaFree(l.d_terms);
        cudaFree(l.d_row_ids);
    }
    cudaFree(r->d_coefs);
    cudaFree(r->d_z);
    cudaFree(r->d_zraw);
    cudaFree(r->d_first_fail);
    delete r;
    c->r1cs = nullptr;
}

// raw little-endian assignment vectors -> Montgomery residues, witness-minor
template <int N>
__global__ void __launch_bounds__(256)
k_r1cs_load_z(const uint8_t* __restrict__ zraw, uint64_t set_stride, uint32_t stride, uint64_t n_vars, uint32_t* __restrict__ z,
              TileGeom g, uint32_t* unreduced_count, FieldParams fp) {
    const uint64_t total = n_vars << g.log2_wt;
    const uint32_t wt_mask = (1u << g.log2_wt) - 1;
    for (uint64_t tid = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; tid < total; tid += (uint64_t)gridDim.x * blockDim.x) {
        uint32_t lane = (uint32_t)tid & wt_mask;
        uint64_t var = tid >> g.log2_wt;
        uint32_t v[N];
#pragma unroll
        for (int k = 0; k < N; k++) v[k] = 0;
        if (lane < g.n_valid) {
            const uint8_t* src = zraw + (uint64_t)(g.batch0 + lane) * set_stride + var * stride;
            bool ge_p = false;
            load_raw_value<N>(v, ge_p, src, stride, fp);
            if (ge_p) atomicAdd(unreduced_count, 1u);
        }
        store_elem<N>(z, (uint32_t)var, lane, g.log2_wt, v);
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// k_r1cs_check: thread <-> (sorted row, assignment lane), lane fastest.
//
// The kernel waits on the z gathers: random 32-byte sectors of a vector far larger than L2, ~1 us away.  Keeping HBM
// busy needs (bandwidth x latency) / 32 B ~ 1100 sectors in flight per SM; a thread that holds its operands in registers
// keeps one or two (round 1: 2480 GB/s = 0.38 of the copy peak, long_scoreboard 5.4, occupancy 33 % at 80 registers).
// Here NOTHING waits in registers: every thread owns two small rings in shared memory, filled by cp.async (LDGSTS),
//     D ring: the {col, tag} descriptors of its next terms   (8-byte coalesced / broadcast loads)
//     G ring: the z limbs those descriptors name             (16-byte gathers, L2 only: .cg)
// and runs a three-deep software pipeline over its term stream, one commit group per term:
//     step s:  wait until group s - GA has landed      (descriptor of term s - GA, limbs of term s - 2 GA)
//              issue the gather of term s - GA, request the descriptor of term s, commit group s
//              consume term s - 2 GA from shared memory (Montgomery multiply-add)
// so GA gathers and GA descriptor loads per thread are in flight while the integer chain runs, across row boundaries
// (the stream continues into the thread's next row), with no registers tied up.  The stream is self-describing: the top
// two bits of a tag mark the last term of A_r, of B_r and of C_r (build_layout writes them into the device copy), so the
// consumer needs no slice header; only the descriptor cursor reads headers, one item ahead.
// ---------------------------------------------------------------------------------------------------------------------
constexpr uint32_t TD_MASK = 0x3FFFFFFFu;  // device tag: low 30 bits = coefficient index | TD_ONE | TD_PAD
constexpr uint32_t TD_PAD = 0x3FFFFFFFu;
constexpr uint32_t TD_ONE = 0x3FFFFFFEu;
constexpr uint32_t M_END_A = 1, M_END_B = 2, M_END_C = 3;  // tag >> 30

#ifndef ZKB_R1CS_GA
#define ZKB_R1CS_GA 3
#endif
#ifndef ZKB_R1CS_LAZY
#define ZKB_R1CS_LAZY 1
#endif
#ifndef ZKB_R1CS_MIN_CTAS
#define ZKB_R1CS_MIN_CTAS (ZKB_R1CS_LAZY ? 3 : 4)  // the 2N + 1 limb accumulator spills under a 64-register cap (profiles/r02j_ab_r1cs_lazy.log)
#endif
constexpr int kR1csThreads = 256;

__device__ __forceinline__ void cp_async_16(uint32_t smem_dst, const void* gmem_src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_dst), "l"(gmem_src) : "memory");
}
template <int BYTES>
__device__ __forceinline__ void cp_async_small(uint32_t smem_dst, const void* gmem_src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], %2;" ::"r"(smem_dst), "l"(gmem_src), "n"(BYTES) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int PENDING>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(PENDING) : "memory"); }
__device__ __forceinline__ uint2 lds64(uint32_t a) {
    uint2 v;
    asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(a));
    return v;
}
__device__ __forceinline__ void sts64(uint32_t a, uint2 v) { asm volatile("st.shared.v2.u32 [%0], {%1, %2};" ::"r"(a), "r"(v.x), "r"(v.y) : "memory"); }
template <int CW>
__device__ __forceinline__ void lds_chunk(uint32_t* o, uint32_t a) {
    if constexpr (CW == 4) asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(o[0]), "=r"(o[1]), "=r"(o[2]), "=r"(o[3]) : "r"(a));
    else if constexpr (CW == 2) asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(o[0]), "=r"(o[1]) : "r"(a));
    else asm volatile("ld.shared.u32 %0, [%1];" : "=r"(o[0]) : "r"(a));
}
template <int CW>
__device__ __forceinline__ void sts_chunk(uint32_t a, const uint32_t* o) {
    if constexpr (CW == 4) asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(a), "r"(o[0]), "r"(o[1]), "r"(o[2]), "r"(o[3]) : "memory");
    else if constexpr (CW == 2) asm volatile("st.shared.v2.u32 [%0], {%1, %2};" ::"r"(a), "r"(o[0]), "r"(o[1]) : "memory");
    else asm volatile("st.shared.u32 [%0], %1;" ::"r"(a), "r"(o[0]) : "memory");
}

// Ring sizes are powers of two so that a ring position is (step & mask): the D ring needs 2 GA + 1 entries (a descriptor
// lives from its request to the consumption of its term), the G ring GA + 1 (limbs live from the gather to the consumption).
template <int N>
struct R1csSmem {
    static constexpr int GA = ZKB_R1CS_GA;
    static constexpr int RD = GA <= 3 ? 8 : 16;
    static constexpr int RG = GA <= 3 ? 4 : 8;
    static_assert(2 * GA + 1 <= RD && GA + 1 <= RG, "rings too small for this look-ahead");
    static constexpr int CW = Elem<N>::CW, NC = Elem<N>::NC, CB = CW * 4;       // chunk: limbs, count, bytes
    static constexpr uint32_t d_bytes = (uint32_t)RD * kR1csThreads * 8;       // [RD][threads] x {col, tag}
    static constexpr uint32_t g_bytes = (uint32_t)RG * NC * kR1csThreads * CB;  // [RG][NC][threads] x chunk
    static constexpr uint32_t a_bytes = (uint32_t)NC * kR1csThreads * CB;       // [NC][threads]: A_r . z, then (A_r . z)(B_r . z), parked while the next LC runs
    static constexpr size_t bytes = (size_t)d_bytes + g_bytes + a_bytes;
};

template <int N>
__global__ void __launch_bounds__(kR1csThreads, ZKB_R1CS_MIN_CTAS)
k_r1cs_check(const uint4* __restrict__ slices, const uint2* __restrict__ terms, const uint32_t* __restrict__ row_ids,
             const uint32_t* __restrict__ coefs, const uint32_t* __restrict__ z, uint64_t n_rows, uint64_t n_slices,
             uint32_t* __restrict__ first_fail, TileGeom g, FieldParams fp) {
    using S = R1csSmem<N>;
    constexpr int GA = S::GA, NC = S::NC, CW = S::CW;
    constexpr uint32_t D_STEP = kR1csThreads * 8, G_STEP = NC * kR1csThreads * S::CB, C_STEP = kR1csThreads * S::CB;
    extern __shared__ uint4 smem_raw[];
    const uint32_t smem0 = (uint32_t)__cvta_generic_to_shared(smem_raw);
    const uint32_t d_base = smem0 + threadIdx.x * 8;
    const uint32_t g_base = smem0 + S::d_bytes + threadIdx.x * S::CB;
    const uint32_t a_base = smem0 + S::d_bytes + S::g_bytes + threadIdx.x * S::CB;
    const uint2 pad_desc = make_uint2(0, TD_PAD);
#pragma unroll
    for (int i = 0; i < S::RD; i++) sts64(d_base + i * D_STEP, pad_desc);  // terms before the first are padding: no prologue

    const uint64_t total = (n_slices * 32) << g.log2_wt;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    const bool single = g.log2_wt == 0;
    uint64_t d_item = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    const uint32_t lane = (uint32_t)d_item & ((1u << g.log2_wt) - 1);  // the same for every item of this thread (stride is a multiple of the tile)
    const uint8_t* z_lane = reinterpret_cast<const uint8_t*>(z) + (size_t)lane * S::CB;
    const uint32_t z_elem = (uint32_t)(NC * S::CB) << g.log2_wt;   // bytes between consecutive variables
    const uint32_t z_chunk = (uint32_t)S::CB << g.log2_wt;         // bytes between the chunks of one variable

    // ---- descriptor cursor: walks this thread's items (tid, tid + stride, ...), K groups each
    bool d_alive = d_item < total;
    uint4 hdr = d_alive ? __ldg(slices + ((d_item >> g.log2_wt) >> 5)) : make_uint4(0, 0, 0, 0);
    const uint2* d_ptr = terms;
    uint32_t d_left = 0;
    auto d_open = [&]() {  // hdr = header of d_item; afterwards hdr = header of the item after it (load in flight)
        d_left = (hdr.y & 0xFFFF) + (hdr.y >> 16) + (hdr.z & 0xFFFF) + (hdr.z >> 16) + (hdr.w & 0xFFFF) + (hdr.w >> 16);
        d_ptr = terms + (size_t)hdr.x * 32 + ((d_item >> g.log2_wt) & 31);
        const uint64_t nxt = d_item + stride;
        if (nxt < total) hdr = __ldg(slices + ((nxt >> g.log2_wt) >> 5));
    };
    if (d_alive) d_open();
    uint64_t c_item = d_item;  // item the consumer is in
    int drain = 0;

    // the linear combination being summed: for 4- and 8-limb fields the plain integer of field_ptx.cuh's lazy reduction (one
    // Montgomery reduction per linear combination, N^2 multiplications per term instead of 2 N^2), else a reduced residue
    constexpr bool LAZY = ZKB_R1CS_LAZY && (N == 4 || N == 8);
    constexpr int NT = LAZY ? 2 * N + 1 : N;
    uint32_t acc[NT];
#pragma unroll
    for (int i = 0; i < NT; i++) acc[i] = 0;
    bool products = false;  // LAZY: the accumulator holds a product (else it is a sum of residues times R: no REDC needed)

    for (uint32_t s = 0;; s++) {
        cp_async_wait<GA - 1>();
        // (1) gather the limbs of term s - GA: its descriptor has landed
        {
            const uint2 t = lds64(d_base + ((s - GA) & (S::RD - 1)) * D_STEP);
            if ((t.y & TD_MASK) != TD_PAD) {
                const uint8_t* src = z_lane + (uint64_t)t.x * z_elem;
                const uint32_t dst = g_base + ((s - GA) & (S::RG - 1)) * G_STEP;
#pragma unroll
                for (int c = 0; c < NC; c++) {
                    if constexpr (S::CB == 16) cp_async_16(dst + c * C_STEP, src + (size_t)c * z_chunk);
                    else cp_async_small<S::CB>(dst + c * C_STEP, src + (size_t)c * z_chunk);
                }
            }
        }
        // (2) request the descriptor of term s
        if (d_alive) {
            cp_async_small<8>(d_base + (s & (S::RD - 1)) * D_STEP, d_ptr);
            d_ptr += 32;
            if (--d_left == 0) {
                d_item += stride;
                d_alive = d_item < total;
                if (d_alive) d_open();
            }
        } else {
            sts64(d_base + (s & (S::RD - 1)) * D_STEP, pad_desc);  // past the last term: padding drains the pipeline
            if (++drain > 2 * GA) break;
        }
        cp_async_commit();
        // (3) consume term s - 2 GA
        const uint2 t = lds64(d_base + ((s - 2 * GA) & (S::RD - 1)) * D_STEP);
        const uint32_t tag = t.y & TD_MASK;
        if (tag != TD_PAD) {
            uint32_t zl[N];
            const uint32_t srcs = g_base + ((s - 2 * GA) & (S::RG - 1)) * G_STEP;
#pragma unroll
            for (int c = 0; c < NC; c++) lds_chunk<CW>(zl + c * CW, srcs + c * C_STEP);
            if (tag == TD_ONE) {
                if constexpr (LAZY) fe_lazy_add_one<N>(acc, zl);
                else fe_add<N>(acc, acc, zl, fp.p);
            } else {
                uint32_t cf[N];
                using V = typename Vec<CW>::T;
                const V* cv = reinterpret_cast<const V*>(coefs) + (size_t)tag * NC;  // a few KB, L1-resident (the gathers bypass L1)
#pragma unroll
                for (int c = 0; c < NC; c++) unpack(__ldg(cv + c), cf + c * CW);
                if constexpr (LAZY) {
                    fe_lazy_mad<N>(acc, zl, cf);
                    products = true;
                } else {
                    uint32_t prod[N];
                    fe_mont_mul<N>(prod, zl, cf, fp.p, fp.n0inv);
                    fe_add<N>(acc, acc, prod, fp.p);
                }
            }
        }
        const uint32_t mark = t.y >> 30;
        if (mark != 0) {
            uint32_t lc[N];  // the finished linear combination, reduced
            if constexpr (LAZY) {
                fe_lazy_finish<N>(lc, acc, fp.p, fp.n0inv, products);
                products = false;
            } else {
#pragma unroll
                for (int i = 0; i < N; i++) lc[i] = acc[i];
            }
            if (mark == M_END_A) {  // park A_r . z in shared memory: the registers serve B_r
#pragma unroll
                for (int c = 0; c < NC; c++) sts_chunk<CW>(a_base + c * C_STEP, lc + c * CW);
            } else if (mark == M_END_B) {  // (aR)(bR)/R = abR takes the parking place: only the accumulator lives across terms
                uint32_t av[N], ab[N];
#pragma unroll
                for (int c = 0; c < NC; c++) lds_chunk<CW>(av + c * CW, a_base + c * C_STEP);
                fe_mont_mul<N>(ab, av, lc, fp.p, fp.n0inv);
#pragma unroll
                for (int c = 0; c < NC; c++) sts_chunk<CW>(a_base + c * C_STEP, ab + c * CW);
            } else {  // abR against cR
                uint32_t ab[N];
#pragma unroll
                for (int c = 0; c < NC; c++) lds_chunk<CW>(ab + c * CW, a_base + c * C_STEP);
                uint32_t diff = 0;
#pragma unroll
                for (int i = 0; i < N; i++) diff |= ab[i] ^ lc[i];
                const uint64_t srow = c_item >> g.log2_wt;
                const bool fail = diff != 0 && srow < n_rows && lane < g.n_valid;  // the last slice may hold padding rows
                report_fail(fail, fail ? __ldg(row_ids + srow) : 0u, first_fail, g.batch0 + lane, single);
                c_item += stride;
            }
#pragma unroll
            for (int i = 0; i < NT; i++) acc[i] = 0;
        }
    }
    cp_async_wait<0>();
}

static unsigned grid_for(uint64_t total, int sm_count, int per_sm);

// persistent grid: as many CTAs as the shared-memory rings allow, every thread streams through its rows
template <int N>
static void launch_r1cs_check(zkb_ctx* c, R1csDev* r, const R1csLayout& L, TileGeom g, const FieldParams& fp) {
    const size_t smem = R1csSmem<N>::bytes;
    static int per_sm = 0;
    static std::atomic<uint64_t> attr_seen{0};
    if (first_on_device(attr_seen))  // per device: a second GPU of the process needs its own opt-in to 56 KB of shared memory
        cudaFuncSetAttribute(k_r1cs_check<N>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (!per_sm) {
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_r1cs_check<N>, kR1csThreads, smem);
        if (per_sm < 1) per_sm = 1;
        if (const char* e = getenv("ZKB_R1CS_CTAS_PER_SM")) per_sm = std::max(1, atoi(e));
        if (getenv("ZKB_DEBUG")) fprintf(stderr, "zkb: k_r1cs_check<%d>: %d CTAs/SM, %zu B of shared memory per CTA\n", N, per_sm, smem);
    }
    unsigned grid = grid_for((L.n_slices * 32) << g.log2_wt, c->sm_count, per_sm);
    // a thread keeps its assignment lane from row to row: the grid stride must be a multiple of the tile width
    const unsigned m = std::max(1u, (1u << g.log2_wt) / kR1csThreads);
    grid = std::max(m, grid / m * m);
    k_r1cs_check<N><<<grid, kR1csThreads, smem, c->stream>>>(L.d_slices, L.d_terms, L.d_row_ids, r->d_coefs, r->d_z, r->n_rows, L.n_slices,
                                                             r->d_first_fail, g, fp);
}

static unsigned grid_for(uint64_t total, int sm_count, int per_sm) {
    uint64_t blocks = (total + 255) / 256;
    uint64_t cap = (uint64_t)sm_count * per_sm;
    if (blocks > cap) blocks = cap;
    if (blocks == 0) blocks = 1;
    return (unsigned)blocks;
}

}  // namespace zkb

#define DISPATCH_N(nlimb, CALL)                        \
    switch (nlimb) {                                   \
        case 1: { constexpr int N = 1; CALL; } break;  \
        case 2: { constexpr int N = 2; CALL; } break;  \
        case 4: { constexpr int N = 4; CALL; } break;  \
        default: { constexpr int N = 8; CALL; } break; \
    }

extern "C" int zkb_r1cs_load(zkb_ctx* c, const zkb_csr* A, const zkb_csr* B, const zkb_csr* C, const uint8_t* coef_table_le,
                             size_t coef_stride, uint64_t n_coefs, uint64_t n_vars) {
    if (!c->prog.field_set) return c->fail(ZKB_E_ARG, "set_field must be called before zkb_r1cs_load");
    if (c->prog.binary) return c->fail(ZKB_E_UNSUPPORTED, "zkb: R1CS over p = 2 is not supported");
    if (A->n_rows != B->n_rows || A->n_rows != C->n_rows) return c->fail(ZKB_E_ARG, "A, B, C must have the same number of rows");
    if (A->n_rows >= 0xFFFFFFE0ull) return c->fail(ZKB_E_UNSUPPORTED, "zkb: more than 2^32 rows");
    if (n_vars == 0 || n_vars >= 0xFFFFFFFFull) return c->fail(ZKB_E_ARG, "n_vars out of range");
    if (n_coefs >= TD_ONE) return c->fail(ZKB_E_ARG, "coefficient table too large (2^30 - 2 entries at most)");
    if (c->has_gpu) CUDA_TRY(c, cudaSetDevice(c->device));
    r1cs_free(c);
    R1csDev* r = new R1csDev();
    c->r1cs = r;
    const uint64_t nr = A->n_rows;
    r->n_rows = nr;
    r->n_vars = n_vars;
    const zkb_csr* M[3] = {A, B, C};
    for (int m = 0; m < 3; m++) {
        uint64_t nnz = M[m]->row_ptr[nr];
        if (nnz >= 0xFFFFFFFFull) return c->fail(ZKB_E_UNSUPPORTED, "zkb: more than 2^32 non-zeros per matrix");
        r->nnz[m] = nnz;
        for (uint64_t i = 0; i <= nr; i++)
            if (M[m]->row_ptr[i] > nnz || (i && M[m]->row_ptr[i] < M[m]->row_ptr[i - 1])) return c->fail(ZKB_E_ARG, "row_ptr is not monotone");
        for (uint64_t e = 0; e < nnz; e++) {
            if (M[m]->col[e] >= n_vars) return c->fail(ZKB_E_SEMANTIC, "The WireId " + std::to_string(M[m]->col[e]) + " has not been defined yet.");  // from_r1cs.rs:90
            if (M[m]->coef_idx[e] >= n_coefs) return c->fail(ZKB_E_ARG, "coefficient index out of range");
        }
    }
    // coefficient table: reduce mod p on the host (empty coefficient = 0, from_r1cs.rs:72-77), Montgomery on device
    const int N = c->prog.nlimb;
    std::vector<uint32_t> limbs((size_t)std::max<uint64_t>(n_coefs, 1) * N, 0);
    std::vector<uint8_t> coef_class(n_coefs, 2);  // 0: zero (term dropped), 1: one, 2: general
    for (uint64_t i = 0; i < n_coefs; i++) {
        BigU v = BigU::from_bytes_le(coef_table_le + i * coef_stride, coef_stride);
        if (v >= c->prog.modulus) v = v.mod(c->prog.modulus);
        v.to_limbs(&limbs[i * N], N);
        coef_class[i] = v.is_zero() ? 0 : v.is_one() ? 1 : 2;
    }
    r->n_coefs = (uint32_t)n_coefs;
    if (c->has_gpu) {
        CUDA_TRY(c, cudaMalloc((void**)&r->d_coefs, limbs.size() * 4));
        CUDA_TRY(c, cudaMemcpyAsync(r->d_coefs, limbs.data(), limbs.size() * 4, cudaMemcpyHostToDevice, c->stream));
        launch_to_mont(N, r->d_coefs, (uint32_t)n_coefs, c->prog.fp, c->stream);
    }

    // keep the system (zero coefficients dropped: they contribute nothing, from_r1cs.rs:72-77; coefficient one tagged)
    for (int m = 0; m < 3; m++) {
        r->h_rp[m].assign(nr + 1, 0);
        r->h_col[m].reserve(r->nnz[m]);
        r->h_tag[m].reserve(r->nnz[m]);
        for (uint64_t row = 0; row < nr; row++) {
            for (uint64_t e = M[m]->row_ptr[row]; e < M[m]->row_ptr[row + 1]; e++) {
                const uint32_t ci = M[m]->coef_idx[e];
                if (coef_class[ci] == 0) continue;
                r->h_col[m].push_back(M[m]->col[e]);
                r->h_tag[m].push_back(coef_class[ci] == 1 ? T_ONE : ci);
            }
            r->h_rp[m][row + 1] = (uint32_t)r->h_col[m].size();
        }
    }
    if (c->has_gpu) CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    return ZKB_OK;
}

// SELL-32-sigma construction of one layout kind (see R1csLayout); uploads it unless the context is host-only
static int build_layout(zkb_ctx* c, R1csDev* r, int kind) {
    R1csLayout& L = r->layout[kind];
    if (L.built) return ZKB_OK;
    const uint64_t nr = r->n_rows;
    const bool split = kind == 0;
    uint64_t sigma = split ? 262144 : 16384;
    if (const char* e = getenv("ZKB_R1CS_SIGMA")) sigma = std::max<uint64_t>(32, (uint64_t)atoll(e) / 32 * 32);
    // class of a term: 2 * matrix + (general ? 1 : 0); without the split everything is "general"
    auto cls = [&](int m, uint32_t tag) { return 2 * m + ((split && tag == T_ONE) ? 0 : 1); };
    std::vector<uint32_t> cls_cnt(std::max<uint64_t>(nr, 1) * 6, 0);
    for (int m = 0; m < 3; m++)
        for (uint64_t row = 0; row < nr; row++)
            for (uint32_t e = r->h_rp[m][row]; e < r->h_rp[m][row + 1]; e++) {
                uint32_t& n = cls_cnt[row * 6 + cls(m, r->h_tag[m][e])];
                if (++n > 0xFFFF) return c->fail(ZKB_E_UNSUPPORTED, "zkb: more than 65535 terms of one kind in a constraint");
            }
    std::vector<uint32_t> order(std::max<uint64_t>(nr, 1));
    for (uint64_t i = 0; i < nr; i++) order[i] = (uint32_t)i;
    for (uint64_t w0 = 0; w0 < nr; w0 += sigma) {
        uint64_t w1 = std::min(nr, w0 + sigma);
        std::stable_sort(order.begin() + w0, order.begin() + w1, [&](uint32_t x, uint32_t y) {
            const uint32_t* cx = &cls_cnt[(size_t)x * 6];
            const uint32_t* cy = &cls_cnt[(size_t)y * 6];
            for (int k = 0; k < 6; k++)
                if (cx[k] != cy[k]) return cx[k] > cy[k];
            return false;
        });
    }
    const uint64_t n_slices = (nr + 31) / 32;
    std::vector<uint4> slices(std::max<uint64_t>(n_slices, 1));
    uint64_t n_groups = 0;
    for (uint64_t s = 0; s < n_slices; s++) {
        uint32_t k[6] = {0, 0, 0, 0, 0, 0};
        for (uint64_t i = s * 32; i < std::min(nr, s * 32 + 32); i++)
            for (int q = 0; q < 6; q++) k[q] = std::max(k[q], cls_cnt[(size_t)order[i] * 6 + q]);
        if (c->has_gpu)  // the device stream marks the end of A_r, B_r, C_r on a term: every matrix owns at least one group
            for (int m = 0; m < 3; m++)
                if (k[2 * m] + k[2 * m + 1] == 0) k[2 * m + 1] = 1;
        slices[s] = make_uint4((uint32_t)n_groups, k[0] | (k[1] << 16), k[2] | (k[3] << 16), k[4] | (k[5] << 16));
        for (int q = 0; q < 6; q++) n_groups += k[q];
        if (n_groups >= (1ull << 32) / 32) return c->fail(ZKB_E_UNSUPPORTED, "zkb: R1CS too large for the sliced layout");
    }
    std::vector<uint2> terms(std::max<uint64_t>(n_groups, 1) * 32, make_uint2(0, T_PAD));
    for (uint64_t s = 0; s < n_slices; s++) {
        const uint32_t packed[3] = {slices[s].y, slices[s].z, slices[s].w};
        uint64_t base[6];  // first group of every class in this slice
        uint64_t gpos = slices[s].x;
        for (int q = 0; q < 6; q++) {
            base[q] = gpos;
            gpos += (packed[q / 2] >> (16 * (q & 1))) & 0xFFFF;
        }
        for (uint64_t i = s * 32; i < std::min(nr, s * 32 + 32); i++) {
            const uint64_t row = order[i];
            uint32_t fill[6] = {0, 0, 0, 0, 0, 0};
            for (int m = 0; m < 3; m++)
                for (uint32_t e = r->h_rp[m][row]; e < r->h_rp[m][row + 1]; e++) {
                    const int q = cls(m, r->h_tag[m][e]);
                    terms[(base[q] + fill[q]++) * 32 + (i & 31)] = make_uint2(r->h_col[m][e], r->h_tag[m][e]);
                }
        }
    }
    L.n_slices = n_slices;
    L.n_groups = n_groups;
    L.built = true;
    if (!c->has_gpu) {  // host-only context: the layout can be inspected, every evaluation call fails with ZKB_E_CUDA
        L.h_slices = std::move(slices);
        L.h_terms = std::move(terms);
        L.h_row_ids = std::move(order);
        return ZKB_OK;
    }
    // device tags: 30-bit payload + end-of-A / end-of-B / end-of-C marker on the last group of each matrix
    for (uint64_t s = 0; s < n_slices; s++) {
        const uint32_t kA = (slices[s].y & 0xFFFF) + (slices[s].y >> 16), kB = (slices[s].z & 0xFFFF) + (slices[s].z >> 16),
                       kC = (slices[s].w & 0xFFFF) + (slices[s].w >> 16);
        const uint64_t g0 = slices[s].x;
        for (uint64_t gi = g0; gi < g0 + kA + kB + kC; gi++) {
            const uint32_t mark = gi == g0 + kA - 1 ? M_END_A : gi == g0 + kA + kB - 1 ? M_END_B : gi == g0 + kA + kB + kC - 1 ? M_END_C : 0;
            for (int l = 0; l < 32; l++) {
                uint32_t& t = terms[gi * 32 + l].y;
                t = (t == T_PAD ? TD_PAD : t == T_ONE ? TD_ONE : t) | (mark << 30);
            }
        }
    }
    CUDA_TRY(c, cudaMalloc((void**)&L.d_slices, slices.size() * sizeof(uint4)));
    CUDA_TRY(c, cudaMalloc((void**)&L.d_terms, terms.size() * sizeof(uint2)));
    CUDA_TRY(c, cudaMalloc((void**)&L.d_row_ids, order.size() * 4));
    CUDA_TRY(c, cudaMemcpy(L.d_slices, slices.data(), slices.size() * sizeof(uint4), cudaMemcpyHostToDevice));
    CUDA_TRY(c, cudaMemcpy(L.d_terms, terms.data(), terms.size() * sizeof(uint2), cudaMemcpyHostToDevice));
    CUDA_TRY(c, cudaMemcpy(L.d_row_ids, order.data(), order.size() * 4, cudaMemcpyHostToDevice));
    return ZKB_OK;
}

extern "C" int zkb_debug_r1cs_layout(zkb_ctx* c, int kind, uint64_t counts[3], uint32_t* slices, uint32_t* terms, uint32_t* row_ids) {
    R1csDev* r = c->r1cs;
    if (!r) return c->fail(ZKB_E_ARG, "zkb_r1cs_load must be called first");
    if (c->has_gpu) return c->fail(ZKB_E_ARG, "zkb_debug_r1cs_layout needs a host-only context (device < 0)");
    if (kind != 0 && kind != 1) return c->fail(ZKB_E_ARG, "layout kind must be 0 or 1");
    int rc = build_layout(c, r, kind);
    if (rc != ZKB_OK) return rc;
    const R1csLayout& L = r->layout[kind];
    counts[0] = L.n_slices;
    counts[1] = L.n_groups;
    counts[2] = r->n_rows;
    if (slices) memcpy(slices, L.h_slices.data(), L.n_slices * sizeof(uint4));
    if (terms) memcpy(terms, L.h_terms.data(), L.n_groups * 32 * sizeof(uint2));
    if (row_ids) memcpy(row_ids, L.h_row_ids.data(), r->n_rows * 4);
    return ZKB_OK;
}

extern "C" int zkb_r1cs_upload(zkb_ctx* c, const uint8_t* z_le, uint64_t z_set_stride, uint32_t value_stride, uint32_t n_batch) {
    R1csDev* r = c->r1cs;
    if (!r) return c->fail(ZKB_E_ARG, "zkb_r1cs_load must be called first");
    if (!c->has_gpu) return c->fail(ZKB_E_CUDA, "no CUDA device in this context (there is no CPU fallback)");
    if (n_batch == 0 || value_stride == 0) return c->fail(ZKB_E_ARG, "n_batch and value_stride must be > 0");
    if (n_batch > 1 && z_set_stride < r->n_vars * value_stride) return c->fail(ZKB_E_ARG, "z_set_stride smaller than one assignment vector");
    // variable 0 is the constant one (from_r1cs.rs:40-42, 52-56)
    for (uint32_t j = 0; j < n_batch; j++) {
        BigU one = BigU::from_bytes_le(z_le + (size_t)j * z_set_stride, value_stride);
        if (!one.is_one()) return c->fail(ZKB_E_FATAL, "value for instance id:0 should be a constant 1");
    }
    CUDA_TRY(c, cudaSetDevice(c->device));
    const size_t eb = (size_t)c->prog.nlimb * 4;
    uint32_t want = 0;
    while (((uint64_t)1 << want) < n_batch) want++;
    size_t free_b = 0, total_b = 0;
    CUDA_TRY(c, cudaMemGetInfo(&free_b, &total_b));
    size_t raw = (size_t)(n_batch > 1 ? z_set_stride * n_batch : r->n_vars * value_stride);
    size_t budget = free_b + r->z_bytes + r->zraw_bytes;
    budget = budget > raw + ((size_t)768 << 20) ? budget - raw - ((size_t)768 << 20) : 0;
    uint32_t l2 = want;
    while (l2 > 0 && r->n_vars * eb * ((size_t)1 << l2) > budget) l2--;
    if (const char* s = getenv("ZKB_TILE_LOG2")) {
        uint32_t f = (uint32_t)atoi(s);
        if (f < l2) l2 = f;
    }
    size_t need = r->n_vars * eb * ((size_t)1 << l2);
    if (need > budget) return c->fail(ZKB_E_CUDA, "assignment vector does not fit in device memory");
    CUDA_TRY(c, cudaEventRecord(c->ev[0], c->stream));
    if (need > r->z_bytes) {
        cudaFree(r->d_z);
        r->d_z = nullptr;
        r->z_bytes = 0;
        CUDA_TRY(c, cudaMalloc((void**)&r->d_z, need));
        r->z_bytes = need;
    }
    if (raw > r->zraw_bytes) {
        cudaFree(r->d_zraw);
        r->d_zraw = nullptr;
        r->zraw_bytes = 0;
        CUDA_TRY(c, cudaMalloc((void**)&r->d_zraw, raw));
        r->zraw_bytes = raw;
    }
    CUDA_TRY(c, cudaMemcpyAsync(r->d_zraw, z_le, raw, cudaMemcpyHostToDevice, c->stream));
    CUDA_TRY(c, cudaEventRecord(c->ev[1], c->stream));
    if (n_batch > r->first_fail_cap) {
        cudaFree(r->d_first_fail);
        r->d_first_fail = nullptr;
        CUDA_TRY(c, cudaMalloc((void**)&r->d_first_fail, (size_t)n_batch * 4));
        r->first_fail_cap = n_batch;
    }
    {
        int rc = build_layout(c, r, l2 < 5 ? 0 : 1);  // first use of this tile width class: build + upload the layout
        if (rc != ZKB_OK) return rc;
    }
    r->z_set_stride = z_set_stride;
    r->stride = value_stride;
    r->n_batch = n_batch;
    r->log2_wt = l2;
    r->uploaded = true;
    return ZKB_OK;
}

extern "C" int zkb_r1cs_run(zkb_ctx* c, zkb_verdict* out) {
    R1csDev* r = c->r1cs;
    if (!r || !r->uploaded) return c->fail(ZKB_E_ARG, "zkb_r1cs_upload must be called first");
    CUDA_TRY(c, cudaSetDevice(c->device));
    const int N = c->prog.nlimb;
    const FieldParams fp = c->prog.fp;
    const uint32_t wt = 1u << r->log2_wt;
    const uint32_t n_tiles = (r->n_batch + wt - 1) / wt;
    uint64_t launches = 0;
    CUDA_TRY(c, cudaEventRecord(c->ev[2], c->stream));
    launch_fill_u32(r->d_first_fail, 0xFFFFFFFFu, r->n_batch, c->sm_count, c->stream);
    CUDA_TRY(c, cudaMemsetAsync(c->d_unreduced, 0, 4, c->stream));
    launches++;
    while (c->tile_ev.size() < 2 * (size_t)n_tiles) {
        cudaEvent_t e;
        cudaEventCreate(&e);
        c->tile_ev.push_back(e);
    }
    for (uint32_t t = 0; t < n_tiles; t++) {
        TileGeom g;
        g.log2_wt = r->log2_wt;
        g.batch0 = t << r->log2_wt;
        g.n_valid = std::min<uint32_t>(wt, r->n_batch - g.batch0);
        g.skip_mask = 0;
        unsigned grid = grid_for(r->n_vars << r->log2_wt, c->sm_count, 256);
        DISPATCH_N(N, (k_r1cs_load_z<N><<<grid, 256, 0, c->stream>>>(r->d_zraw, r->z_set_stride, r->stride, r->n_vars, r->d_z, g,
                                                                     c->d_unreduced, fp)));
        cudaEventRecord(c->tile_ev[2 * t], c->stream);
        const R1csLayout& L = r->layout[r->log2_wt < 5 ? 0 : 1];
        DISPATCH_N(N, (launch_r1cs_check<N>(c, r, L, g, fp)));
        cudaEventRecord(c->tile_ev[2 * t + 1], c->stream);
        launches += 2;
    }
    {
        int rcb = ctx_result_buffer(c, (size_t)r->n_batch + 1);
        if (rcb != ZKB_OK) return rcb;
    }
    CUDA_TRY(c, cudaMemcpyAsync(c->h_res, r->d_first_fail, (size_t)r->n_batch * 4, cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(c, cudaMemcpyAsync(c->h_res + r->n_batch, c->d_unreduced, 4, cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(c, cudaEventRecord(c->ev[3], c->stream));
    CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    CUDA_TRY(c, cudaGetLastError());
    float ms = 0, lv = 0;
    cudaEventElapsedTime(&ms, c->ev[2], c->ev[3]);
    for (uint32_t t = 0; t < n_tiles; t++) {
        float x = 0;
        cudaEventElapsedTime(&x, c->tile_ev[2 * t], c->tile_ev[2 * t + 1]);
        lv += x;
    }
    c->timing.total_ms = ms;
    c->timing.levels_ms = lv;  // the check kernel
    c->timing.load_ms = ms - lv;
    c->timing.h2d_ms = 0;
    c->timing.level_launches = n_tiles;
    c->timing.kernel_launches = launches;
    // values >= p are legal inputs for the reference (kept raw, reduced by the first Mul/Add they meet):
    // every z value passes through Mul(var, const) or the LC additions, so residues are exact here.
    if (out)
        for (uint32_t j = 0; j < r->n_batch; j++) {
            uint32_t f = c->h_res[j];
            memset(&out[j], 0, sizeof(zkb_verdict));
            out[j].ok = f == 0xFFFFFFFFu;
            out[j].first_fail_seq = f == 0xFFFFFFFFu ? UINT64_MAX : f;
        }
    return ZKB_OK;
}

extern "C" int zkb_r1cs_check(zkb_ctx* c, const uint8_t* z_le, uint64_t z_set_stride, uint32_t value_stride, uint32_t n_batch,
                              zkb_verdict* out) {
    int rc = zkb_r1cs_upload(c, z_le, z_set_stride, value_stride, n_batch);
    if (rc != ZKB_OK) return rc;
    rc = zkb_r1cs_run(c, out);
    if (rc != ZKB_OK) return rc;
    float h2d = 0, total = 0;
    cudaEventElapsedTime(&h2d, c->ev[0], c->ev[1]);
    cudaEventElapsedTime(&total, c->ev[0], c->ev[3]);
    c->timing.h2d_ms = h2d;
    c->timing.total_ms = total;
    return ZKB_OK;
}
