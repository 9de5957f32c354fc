// Debug / measurement entry points (not on the product path):
//   zkb_debug_field_ops         element-wise field ops on the device, both the PTX carry-chain product and the
//                               portable CIOS product, so tests can compare them with Python integers
//   zkb_debug_gather_throughput random 32-byte gathers per second from a table larger than L2: the ceiling of the R1CS check
//   zkb_debug_field_throughput  register-resident Montgomery products / modular additions per second: the
//                               integer-pipe ceiling of the level kernel (DESIGN.md section 4)
#include <algorithm>
#include <vector>

#include "context.h"
#include "device_util.cuh"
#include "kernels.cuh"

using namespace zkb;

#define CUDA_TRY(c, expr)                                                                              \
    do {                                                                                               \
        cudaError_t e__ = (expr);                                                                      \
        if (e__ != cudaSuccess)                                                                        \
            return (c)->fail(ZKB_E_CUDA, std::string("CUDA error: ") + cudaGetErrorString(e__) + " at " #expr); \
    } while (0)

namespace {

// op: 0 add, 1 mont_mul (the product of the level kernels, FORM = the field's mul_form), 2 mont_mul portable,
//     3 lazy reduction: REDC(a b + a b + a b + b R) = 3 mont_mul(a, b) + b,  4: REDC(a R + b R) = a + b  (N = 4, 8 only)
template <int N, uint32_t FORM>
__global__ void k_field_ops(int op, const uint32_t* a, const uint32_t* b, uint32_t* r, uint64_t n, FieldParams fp) {
    uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t x[N], y[N], z[N];
#pragma unroll
    for (int k = 0; k < N; k++) {
        x[k] = a[i * N + k];
        y[k] = b[i * N + k];
    }
    if (op == 0) fe_add<N>(z, x, y, fp.p);
    else if (op == 1) fe_mont_mul_form<N, FORM>(z, x, y, fp.p, fp.n0inv);
    else if (op == 2) fe_mont_mul_portable<N>(z, x, y, fp.p, fp.n0inv);
    else if constexpr (N == 4 || N == 8) {
        uint32_t T[2 * N + 1];
#pragma unroll
        for (int k = 0; k < 2 * N + 1; k++) T[k] = 0;
        if (op == 3) {
            fe_lazy_mad<N>(T, x, y);
            fe_lazy_mad<N>(T, x, y);
            fe_lazy_add_one<N>(T, y);
            fe_lazy_mad<N>(T, x, y);
        } else if (op == 4) {
            fe_lazy_add_one<N>(T, x);
            fe_lazy_add_one<N>(T, y);
        } else if (op == 5) {  // one product
            fe_lazy_mad<N>(T, x, y);
        } else if (op == 6) {  // REDC of the N-limb integer a alone
#pragma unroll
            for (int k = 0; k < N; k++) T[k] = x[k];
        } else {               // op 7: low half of the plain product (no reduction): checks fe_mul_wide limb by limb
            uint32_t P[2 * N];
            fe_mul_wide<N>(P, x, y);
#pragma unroll
            for (int k = 0; k < N; k++) z[k] = op == 7 ? P[k] : P[N + k];
        }
        if (op >= 7) {
#pragma unroll
            for (int k = 0; k < N; k++) r[i * N + k] = z[k];
            return;
        }
        fe_lazy_finish<N>(z, T, fp.p, fp.n0inv);
    } else {
#pragma unroll
        for (int k = 0; k < N; k++) z[k] = 0;
    }
#pragma unroll
    for (int k = 0; k < N; k++) r[i * N + k] = z[k];
}

// a chain of dependent products per thread (x <- x*y), operands in registers: no memory traffic
template <int N, uint32_t FORM>
__global__ void __launch_bounds__(256) k_field_throughput(int op, uint32_t iters, uint32_t* sink, FieldParams fp) {
    uint32_t x[N], y[N];
#pragma unroll
    for (int k = 0; k < N; k++) {
        x[k] = (threadIdx.x * 2654435761u + k * 40503u + blockIdx.x) & (k == N - 1 ? 0x0FFFFFFFu : 0xFFFFFFFFu);
        y[k] = (threadIdx.x * 97u + k * 7919u + 12345u) & (k == N - 1 ? 0x0FFFFFFFu : 0xFFFFFFFFu);
    }
    for (uint32_t i = 0; i < iters; i++) {
        uint32_t z[N];
        if (op == 0) fe_add<N>(z, x, y, fp.p);
        else fe_mont_mul_form<N, FORM>(z, x, y, fp.p, fp.n0inv);
#pragma unroll
        for (int k = 0; k < N; k++) x[k] = z[k];
    }
    uint32_t acc = 0;
#pragma unroll
    for (int k = 0; k < N; k++) acc ^= x[k];
    if (acc == 0x12345678u) sink[0] = acc;  // keep the chain alive
}

// random 32-byte gathers (two 16-byte loads of one sector) from a table far larger than L2, 8 independent gathers in
// flight per thread: the ceiling of any kernel whose traffic is z[col] look-ups (k_r1cs_check with one assignment)
__global__ void __launch_bounds__(256) k_gather_throughput(const uint4* __restrict__ table, uint64_t n_elems, uint32_t iters, uint32_t* sink) {
    uint64_t x = (blockIdx.x * 256ull + threadIdx.x) * 0x9E3779B97F4A7C15ull + 0x1234567ull;
    uint4 acc = make_uint4(0, 0, 0, 0);
    for (uint32_t i = 0; i < iters; i++) {
        uint4 v[16];
#pragma unroll
        for (int k = 0; k < 8; k++) {
            x = x * 6364136223846793005ull + 1442695040888963407ull;
            const uint64_t e = (uint64_t)(((x >> 32) * n_elems) >> 32);
            v[2 * k] = __ldcg(table + 2 * e);
            v[2 * k + 1] = __ldcg(table + 2 * e + 1);
        }
#pragma unroll
        for (int k = 0; k < 16; k++) {
            acc.x ^= v[k].x;
            acc.y ^= v[k].y;
            acc.z ^= v[k].z;
            acc.w ^= v[k].w;
        }
    }
    if ((acc.x ^ acc.y ^ acc.z ^ acc.w) == 0x12345678u) sink[0] = acc.x;
}

}  // namespace

// N and the product's form (FieldParams::mul_form), as launch_level chooses them
#define DISPATCH_N(fp, CALL)                                                                                   \
    if ((fp).nlimb == 8 && (fp).mul_form == kMulFormLow64) {                                                   \
        constexpr int N = 8;                                                                                   \
        constexpr uint32_t FORM = kMulFormLow64;                                                               \
        CALL;                                                                                                  \
    } else {                                                                                                   \
        constexpr uint32_t FORM = kMulFormGeneric;                                                             \
        switch ((fp).nlimb) {                                                                                  \
            case 1: { constexpr int N = 1; CALL; } break;                                                      \
            case 2: { constexpr int N = 2; CALL; } break;                                                      \
            case 4: { constexpr int N = 4; CALL; } break;                                                      \
            default: { constexpr int N = 8; CALL; } break;                                                     \
        }                                                                                                      \
    }

extern "C" int zkb_debug_field_ops(zkb_ctx* c, int op, const uint32_t* a, const uint32_t* b, uint32_t* r, uint64_t n) {
    if (!c->prog.field_set || c->prog.binary) return c->fail(ZKB_E_ARG, "set an odd field first");
    if (!c->has_gpu) return c->fail(ZKB_E_CUDA, "no CUDA device in this context (there is no CPU fallback)");
    CUDA_TRY(c, cudaSetDevice(c->device));
    const int N = c->prog.nlimb;
    size_t bytes = (size_t)n * N * 4;
    uint32_t *da = nullptr, *db = nullptr, *dr = nullptr;
    CUDA_TRY(c, cudaMalloc((void**)&da, bytes));
    CUDA_TRY(c, cudaMalloc((void**)&db, bytes));
    CUDA_TRY(c, cudaMalloc((void**)&dr, bytes));
    CUDA_TRY(c, cudaMemcpyAsync(da, a, bytes, cudaMemcpyHostToDevice, c->stream));
    CUDA_TRY(c, cudaMemcpyAsync(db, b, bytes, cudaMemcpyHostToDevice, c->stream));
    const FieldParams fp = c->prog.fp;
    DISPATCH_N(fp, (k_field_ops<N, FORM><<<(unsigned)((n + 127) / 128), 128, 0, c->stream>>>(op, da, db, dr, n, fp)));
    CUDA_TRY(c, cudaMemcpyAsync(r, dr, bytes, cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    cudaFree(da);
    cudaFree(db);
    cudaFree(dr);
    return ZKB_OK;
}

extern "C" int zkb_debug_field_throughput(zkb_ctx* c, int op, uint32_t iters, double* ops_per_second) {
    if (!c->prog.field_set || c->prog.binary) return c->fail(ZKB_E_ARG, "set an odd field first");
    if (!c->has_gpu) return c->fail(ZKB_E_CUDA, "no CUDA device in this context (there is no CPU fallback)");
    CUDA_TRY(c, cudaSetDevice(c->device));
    const FieldParams fp = c->prog.fp;
    uint32_t* sink = nullptr;
    CUDA_TRY(c, cudaMalloc((void**)&sink, 4));
    const unsigned grid = (unsigned)c->sm_count * 8;
    float best = 1e30f;
    for (int rep = 0; rep < 4; rep++) {
        CUDA_TRY(c, cudaEventRecord(c->ev[0], c->stream));
        DISPATCH_N(fp, (k_field_throughput<N, FORM><<<grid, 256, 0, c->stream>>>(op, iters, sink, fp)));
        CUDA_TRY(c, cudaEventRecord(c->ev[1], c->stream));
        CUDA_TRY(c, cudaStreamSynchronize(c->stream));
        float ms = 0;
        cudaEventElapsedTime(&ms, c->ev[0], c->ev[1]);
        if (rep > 0) best = std::min(best, ms);
    }
    cudaFree(sink);
    *ops_per_second = (double)grid * 256.0 * iters / (best * 1e-3);
    return ZKB_OK;
}

extern "C" int zkb_debug_gather_throughput(zkb_ctx* c, uint64_t table_bytes, uint32_t iters, double* bytes_per_second) {
    if (!c->has_gpu) return c->fail(ZKB_E_CUDA, "no CUDA device in this context (there is no CPU fallback)");
    if (table_bytes < 64 || iters == 0) return c->fail(ZKB_E_ARG, "table_bytes >= 64 and iters > 0");
    CUDA_TRY(c, cudaSetDevice(c->device));
    uint4* table = nullptr;
    uint32_t* sink = nullptr;
    CUDA_TRY(c, cudaMalloc((void**)&table, table_bytes));
    CUDA_TRY(c, cudaMalloc((void**)&sink, 4));
    CUDA_TRY(c, cudaMemsetAsync(table, 0x5A, table_bytes, c->stream));
    const unsigned grid = (unsigned)c->sm_count * 8;
    float best = 1e30f;
    for (int rep = 0; rep < 4; rep++) {
        CUDA_TRY(c, cudaEventRecord(c->ev[0], c->stream));
        k_gather_throughput<<<grid, 256, 0, c->stream>>>(table, table_bytes / 32, iters, sink);
        CUDA_TRY(c, cudaEventRecord(c->ev[1], c->stream));
        CUDA_TRY(c, cudaStreamSynchronize(c->stream));
        float ms = 0;
        cudaEventElapsedTime(&ms, c->ev[0], c->ev[1]);
        if (rep > 0) best = std::min(best, ms);
    }
    cudaFree(table);
    cudaFree(sink);
    *bytes_per_second = (double)grid * 256.0 * iters * 8.0 * 32.0 / (best * 1e-3);
    return ZKB_OK;
}

// microseconds per barrier (kind 0: cooperative_groups grid.sync(), 1: the counter barrier k_levels_coop uses, 2: the hardware
// barrier of one 8-CTA cluster) with `blocks` CTAs of 256 threads: n_levels x this is the latency floor of a single-witness
// statement evaluated in one launch (SURVEY.md section 8d, config C2)
extern "C" int zkb_debug_barrier_cost(zkb_ctx* c, int kind, uint32_t blocks, uint32_t n_barriers, double* us_per_barrier) {
    if (!c->has_gpu) return c->fail(ZKB_E_CUDA, "no CUDA device in this context (there is no CPU fallback)");
    if (kind < 0 || kind > 2 || n_barriers == 0) return c->fail(ZKB_E_ARG, "kind in 0..2 and n_barriers > 0");
    CUDA_TRY(c, cudaSetDevice(c->device));
    if (blocks == 0) blocks = (uint32_t)c->sm_count;
    float us = 0;
    CUDA_TRY(c, measure_barrier_cost(kind, blocks, n_barriers, c->d_barrier, &c->barrier_epoch, c->stream, c->ev[0], c->ev[1], &us));
    *us_per_barrier = us;
    return ZKB_OK;
}
