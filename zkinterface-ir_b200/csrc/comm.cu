// Multi-GPU behind the C ABI (include/zkb.h section 7; SURVEY.md section 8b `zkb_comm_init`, section 8e).
//
// The reference is one thread (no analogue to cite beyond the Evaluator it parallelises: evaluator.rs:191-230 runs one
// witness at a time).  The path shards over independent witnesses: one levelized program, replicated; rank r evaluates a
// contiguous block of the batch; the only exchange is ONE MIN all-reduce of the per-witness first_fail vector
// (TRUE = 0xFFFFFFFF), i.e. an AND of the verdict bits.
//
//   * the program is levelized ONCE, on the root rank; zkb_comm_broadcast_program ships the device plan (gate descriptors,
//     assertion table, input loads, Montgomery constants, level offsets, the value -> slot tables read-back consults)
//     device-to-device with ncclBroadcast, plus a small host table (level offsets, input loads, assertion wire ids);
//   * ranks are contexts: N contexts of one process (zkb_comm_init: ncclCommInitAll, one host thread per device in
//     zkb_evaluate_sharded) or one context per process (zkb_comm_unique_id + zkb_comm_init_rank: torchrun / MPI style);
//   * NCCL is bound at run time from libnccl.so.2 (the copy the process already holds, e.g. PyTorch's, else the system
//     one): libzkb.so has no link-time dependency on it and single-GPU users never load it;
//   * contexts of one process that SHARE a device cannot form an NCCL communicator ("duplicate GPU"); they get the
//     in-process transport below (peer copies on the contexts' streams + a MIN kernel).  It exists so that the replica
//     path is testable on a one-GPU box; distinct devices always go through NCCL.
#include <dlfcn.h>
#include <nccl.h>
#include <stdio.h>
#include <string.h>

#include <chrono>
#include <condition_variable>
#include <memory>
#include <mutex>
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

// ---------------------------------------------------------------------------------------------- NCCL, bound at run time
struct NcclApi {
    void* handle = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommInitAll)(ncclComm_t*, int, const int*) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Broadcast)(const void*, void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    const char* (*GetErrorString)(ncclResult_t) = nullptr;
    ncclResult_t (*GetVersion)(int*) = nullptr;
    std::string error;
};

static NcclApi* nccl_api() {
    static NcclApi api;
    static std::once_flag once;
    std::call_once(once, [] {
        const char* names[] = {getenv("ZKB_NCCL_LIB"), "libnccl.so.2", "libnccl.so"};
        for (const char* n : names) {
            if (!n || !*n) continue;
            api.handle = dlopen(n, RTLD_NOW | RTLD_NOLOAD);  // the copy this process already holds, if any
            if (!api.handle) api.handle = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
            if (api.handle) break;
        }
        if (!api.handle) {
            api.error = std::string("zkb: NCCL is not available (dlopen libnccl.so.2: ") + (dlerror() ? dlerror() : "?") + ")";
            return;
        }
#define BIND(field, sym)                                                                 \
    *(void**)(&api.field) = dlsym(api.handle, sym);                                      \
    if (!api.field && api.error.empty()) api.error = std::string("zkb: libnccl lacks ") + sym
        BIND(GetUniqueId, "ncclGetUniqueId");
        BIND(CommInitRank, "ncclCommInitRank");
        BIND(CommInitAll, "ncclCommInitAll");
        BIND(CommDestroy, "ncclCommDestroy");
        BIND(AllReduce, "ncclAllReduce");
        BIND(Broadcast, "ncclBroadcast");
        BIND(GroupStart, "ncclGroupStart");
        BIND(GroupEnd, "ncclGroupEnd");
        BIND(GetErrorString, "ncclGetErrorString");
        BIND(GetVersion, "ncclGetVersion");
#undef BIND
    });
    return &api;
}

#define NCCL_TRY(c, api, expr)                                                                              \
    do {                                                                                                    \
        ncclResult_t r__ = (expr);                                                                          \
        if (r__ != ncclSuccess)                                                                             \
            return (c)->fail(ZKB_E_CUDA, std::string("NCCL error: ") + (api)->GetErrorString(r__) + " at " #expr); \
    } while (0)

// ---------------------------------------------------------------------------------------------- in-process transport
// N contexts of one process, one host thread each inside a collective.  A collective is: everybody publishes its buffer,
// meets at the barrier, copies, meets again.
struct LocalGroup {
    int size = 0;
    std::mutex mu;
    std::condition_variable cv;
    int waiting = 0;
    uint64_t generation = 0;
    std::vector<void*> buf;      // per rank: the buffer it brought to the running collective
    std::vector<int> device;
    void barrier() {
        std::unique_lock<std::mutex> lk(mu);
        uint64_t gen = generation;
        if (++waiting == size) {
            waiting = 0;
            generation++;
            cv.notify_all();
        } else {
            cv.wait(lk, [&] { return generation != gen; });
        }
    }
};

struct CommState {
    int rank = 0, size = 1;
    ncclComm_t nccl = nullptr;
    std::shared_ptr<LocalGroup> local;
    uint32_t* d_scratch = nullptr;  // local transport: a peer's vector during the MIN reduction
    size_t scratch_cap = 0;
    uint64_t program_generation = 0;  // bumped by every broadcast this rank took part in
};

__global__ void k_min_u32(uint32_t* __restrict__ dst, const uint32_t* __restrict__ src, size_t n) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        dst[i] = min(dst[i], src[i]);
}

void comm_free(zkb_ctx* c) {
    if (!c->comm) return;
    if (c->comm->nccl) nccl_api()->CommDestroy(c->comm->nccl);
    if (c->comm->d_scratch) cudaFree(c->comm->d_scratch);
    delete c->comm;
    c->comm = nullptr;
}

static int comm_broadcast(zkb_ctx* c, void* d_buf, size_t bytes, int root) {
    CommState* cm = c->comm;
    if (bytes == 0 || cm->size == 1) return ZKB_OK;
    if (cm->nccl) {
        NcclApi* api = nccl_api();
        NCCL_TRY(c, api, api->Broadcast(d_buf, d_buf, bytes, ncclUint8, root, cm->nccl, c->stream));
        return ZKB_OK;
    }
    LocalGroup* g = cm->local.get();
    CUDA_TRY(c, cudaStreamSynchronize(c->stream));  // root: the data is complete; peers: the buffer is idle
    g->buf[cm->rank] = d_buf;
    g->barrier();
    cudaError_t e = cudaSuccess;
    if (cm->rank != root) {
        e = cudaMemcpyPeerAsync(d_buf, c->device, g->buf[root], g->device[root], bytes, c->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    }
    g->barrier();  // nobody re-uses or frees its buffer before every copy has landed
    if (e != cudaSuccess) return c->fail(ZKB_E_CUDA, std::string("CUDA error in the in-process broadcast: ") + cudaGetErrorString(e));
    return ZKB_OK;
}

int comm_allreduce_min_u32(zkb_ctx* c, uint32_t* d_buf, size_t n) {
    CommState* cm = c->comm;
    if (!cm) return c->fail(ZKB_E_ARG, "this context is not part of a communicator (zkb_comm_init / zkb_comm_init_rank)");
    if (cm->size == 1 || n == 0) return ZKB_OK;
    if (cm->nccl) {
        NcclApi* api = nccl_api();
        NCCL_TRY(c, api, api->AllReduce(d_buf, d_buf, n, ncclUint32, ncclMin, cm->nccl, c->stream));
        return ZKB_OK;
    }
    LocalGroup* g = cm->local.get();
    cudaError_t e = cudaStreamSynchronize(c->stream);
    g->buf[cm->rank] = d_buf;
    g->barrier();
    if (cm->rank == 0 && e == cudaSuccess) {
        if (n > cm->scratch_cap) {
            if (cm->d_scratch) cudaFree(cm->d_scratch);
            cm->d_scratch = nullptr;
            cm->scratch_cap = 0;
            e = cudaMalloc((void**)&cm->d_scratch, n * 4);
            if (e == cudaSuccess) cm->scratch_cap = n;
        }
        for (int r = 1; r < cm->size && e == cudaSuccess; r++) {
            e = cudaMemcpyPeerAsync(cm->d_scratch, c->device, g->buf[r], g->device[r], n * 4, c->stream);
            if (e == cudaSuccess) k_min_u32<<<(unsigned)std::min<size_t>((n + 255) / 256, 1024), 256, 0, c->stream>>>(d_buf, cm->d_scratch, n);
        }
        if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    }
    g->barrier();
    if (cm->rank != 0 && e == cudaSuccess) {
        e = cudaMemcpyPeerAsync(d_buf, c->device, g->buf[0], g->device[0], n * 4, c->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    }
    g->barrier();
    if (e != cudaSuccess) return c->fail(ZKB_E_CUDA, std::string("CUDA error in the in-process all-reduce: ") + cudaGetErrorString(e));
    return ZKB_OK;
}

static int comm_warm_up(zkb_ctx* c) {
    CUDA_TRY(c, cudaSetDevice(c->device));
    uint32_t* d = nullptr;
    CUDA_TRY(c, cudaMalloc((void**)&d, 256));
    CUDA_TRY(c, cudaMemsetAsync(d, 0xFF, 256, c->stream));
    int rc = comm_allreduce_min_u32(c, d, 64);
    if (rc == ZKB_OK) rc = comm_broadcast(c, d, 256, 0);
    cudaError_t e = cudaStreamSynchronize(c->stream);
    cudaFree(d);
    if (rc == ZKB_OK && e != cudaSuccess) return c->fail(ZKB_E_CUDA, std::string("CUDA error: ") + cudaGetErrorString(e));
    return rc;
}

// ---------------------------------------------------------------------------------------------- program replica
// What a peer needs on the HOST to launch the plan, to answer zkb_assert_info / zkb_get_stats and to read values back.
struct ReplicaHeader {
    uint64_t magic;
    uint64_t blob_bytes;
    uint64_t n_ops, n_loads, n_consts, n_values, n_asserts, n_levels;
    uint64_t n_raw_ops, algo_bytes_per_witness, n_reused_slots, ir_gates;
    uint64_t cb_count[CB_KINDS];
    uint64_t n_dev_ops[D_OPS];
    uint64_t modulus_len, pending_len, const_raw_bytes;
    uint64_t n_group_descs, n_group_ops, n_group_tables, n_depth_off, group_regs, callout_slot0, n_callouts, n_group_hints;  // call groups (program.h)
    uint32_t n_slots, max_level_ops, n_instance, n_witness;
    uint32_t nlimb, binary, is_boolean, has_pending, keep_all, const_raw_stride, has_const_flags, pad;
    FieldParams fp;
};
constexpr uint64_t kReplicaMagic = 0x7a6b625f7265706cull;  // "zkb_repl"

template <class T>
static void put(std::vector<uint8_t>& blob, const T* p, size_t n) {
    const uint8_t* b = (const uint8_t*)p;
    blob.insert(blob.end(), b, b + n * sizeof(T));
    blob.resize((blob.size() + 7) & ~(size_t)7);
}
template <class T>
static void get(const uint8_t*& cur, std::vector<T>& v, size_t n) {
    v.resize(n);
    if (n) memcpy(v.data(), cur, n * sizeof(T));
    cur += (n * sizeof(T) + 7) & ~(size_t)7;
}

template <class T>
static int bcast_array(zkb_ctx* c, T*& d_ptr, size_t n, int root, bool is_root) {
    if (!is_root) {
        if (d_ptr) cudaFree(d_ptr);
        d_ptr = nullptr;
        if (n) CUDA_TRY(c, cudaMalloc((void**)&d_ptr, n * sizeof(T)));
    }
    return comm_broadcast(c, d_ptr, n * sizeof(T), root);
}

static int broadcast_program(zkb_ctx* c, int root) {
    CommState* cm = c->comm;
    const bool is_root = cm->rank == root;
    if (is_root && !c->finalized) return c->fail(ZKB_E_ARG, "zkb_comm_broadcast_program: the root's program is not finalized");
    if (!is_root && c->finalized && !c->is_replica)
        return c->fail(ZKB_E_ARG, "zkb_comm_broadcast_program: this context holds a program of its own");
    CUDA_TRY(c, cudaSetDevice(c->device));
    NvtxRange r_b("zkb:program_broadcast");
    const bool dbg = getenv("ZKB_DEBUG") != nullptr;
    auto t_start = std::chrono::steady_clock::now();
    auto lap = [&](const char* what) {
        if (!dbg) return;
        auto now = std::chrono::steady_clock::now();
        fprintf(stderr, "zkb: rank %d broadcast %-14s %8.2f ms\n", cm->rank, what, std::chrono::duration<double, std::milli>(now - t_start).count());
        t_start = now;
    };
    Program& p = c->prog;
    Plan& pl = c->plan;
    ReplicaHeader h;
    std::vector<uint8_t> blob;
    std::vector<uint8_t> const_raw_flat;
    if (is_root) {
        memset(&h, 0, sizeof h);
        h.magic = kReplicaMagic;
        h.n_ops = c->is_replica ? c->replica_n_ops : pl.ops.size();
        h.n_loads = pl.loads.size();
        h.n_consts = p.n_consts();
        h.n_values = c->is_replica ? c->replica_n_values : p.kind.size();
        h.n_asserts = p.asserts.size();
        h.n_levels = pl.n_levels;
        h.n_raw_ops = pl.n_raw_ops;
        h.algo_bytes_per_witness = pl.algo_bytes_per_witness;
        h.n_reused_slots = pl.n_reused_slots;
        h.ir_gates = p.ir_gates;
        memcpy(h.cb_count, p.cb_count, sizeof h.cb_count);
        memcpy(h.n_dev_ops, pl.n_dev_ops, sizeof h.n_dev_ops);
        h.modulus_len = p.modulus_le.size();
        h.pending_len = c->has_pending ? c->pending_error.size() : 0;
        h.n_slots = pl.n_slots;
        h.max_level_ops = pl.max_level_ops;
        h.n_instance = p.n_instance;
        h.n_witness = p.n_witness;
        h.nlimb = (uint32_t)p.nlimb;
        h.binary = p.binary;
        h.is_boolean = c->is_boolean;
        h.has_pending = c->has_pending;
        h.keep_all = c->keep_all;
        h.const_raw_stride = c->const_raw_stride;
        h.has_const_flags = c->d_const_flags != nullptr;
        h.fp = p.fp;
        // raw bytes of the unreduced constants (read-back reports them as the reference holds them): length-prefixed
        for (const auto& r : p.const_raw) {
            uint32_t len = (uint32_t)r.size();
            const_raw_flat.insert(const_raw_flat.end(), (uint8_t*)&len, (uint8_t*)&len + 4);
            const_raw_flat.insert(const_raw_flat.end(), r.begin(), r.end());
        }
        h.const_raw_bytes = const_raw_flat.size();
        put(blob, pl.level_off.data(), pl.level_off.size());
        put(blob, pl.level_rare.data(), pl.level_rare.size());
        put(blob, pl.loads.data(), pl.loads.size());
        put(blob, p.asserts.data(), p.asserts.size());
        put(blob, p.const_limbs.data(), p.const_limbs.size());
        put(blob, p.const_unreduced.data(), p.const_unreduced.size());
        put(blob, const_raw_flat.data(), const_raw_flat.size());
        put(blob, p.modulus_le.data(), p.modulus_le.size());
        put(blob, c->pending_error.data(), (size_t)h.pending_len);
        h.n_group_descs = pl.group_descs.size();
        h.n_group_ops = pl.group_ops.size();
        h.n_group_tables = pl.group_tables.size();
        h.n_depth_off = pl.depth_off.size();
        h.n_group_hints = pl.group_hints.size();
        h.group_regs = pl.group_regs;
        h.callout_slot0 = pl.callout_slot0;
        h.n_callouts = pl.n_callouts;
        put(blob, pl.group_descs.data(), pl.group_descs.size());
        put(blob, pl.group_ops.data(), pl.group_ops.size());
        put(blob, pl.group_tables.data(), pl.group_tables.size());
        put(blob, pl.depth_off.data(), pl.depth_off.size());
        put(blob, pl.group_hints.data(), pl.group_hints.size());
        put(blob, pl.hint_off.data(), pl.hint_off.size());
        h.blob_bytes = blob.size();
    }
    // 1. the fixed-size header
    uint8_t* d_stage = nullptr;
    CUDA_TRY(c, cudaMalloc((void**)&d_stage, sizeof h));
    if (is_root) CUDA_TRY(c, cudaMemcpyAsync(d_stage, &h, sizeof h, cudaMemcpyHostToDevice, c->stream));
    int rc = comm_broadcast(c, d_stage, sizeof h, root);
    if (rc == ZKB_OK && !is_root) {
        cudaError_t e = cudaMemcpyAsync(&h, d_stage, sizeof h, cudaMemcpyDeviceToHost, c->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
        if (e != cudaSuccess) rc = c->fail(ZKB_E_CUDA, std::string("CUDA error: ") + cudaGetErrorString(e));
        else if (h.magic != kReplicaMagic) rc = c->fail(ZKB_E_CUDA, "zkb_comm_broadcast_program: bad header (ranks out of step?)");
    } else if (rc == ZKB_OK) {
        cudaStreamSynchronize(c->stream);
    }
    cudaFree(d_stage);
    if (rc != ZKB_OK) return rc;
    lap("header");
    // 2. the host tables, staged through device memory
    uint8_t* d_blob = nullptr;
    CUDA_TRY(c, cudaMalloc((void**)&d_blob, std::max<size_t>(h.blob_bytes, 16)));
    if (is_root) CUDA_TRY(c, cudaMemcpyAsync(d_blob, blob.data(), h.blob_bytes, cudaMemcpyHostToDevice, c->stream));
    rc = comm_broadcast(c, d_blob, h.blob_bytes, root);
    if (rc == ZKB_OK && !is_root) {
        blob.resize(h.blob_bytes);
        cudaError_t e = cudaMemcpyAsync(blob.data(), d_blob, h.blob_bytes, cudaMemcpyDeviceToHost, c->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
        if (e != cudaSuccess) rc = c->fail(ZKB_E_CUDA, std::string("CUDA error: ") + cudaGetErrorString(e));
    } else if (rc == ZKB_OK) {
        cudaStreamSynchronize(c->stream);
    }
    cudaFree(d_blob);
    if (rc != ZKB_OK) return rc;
    lap("host tables");
    if (!is_root) {
        p = Program();
        pl = Plan();
        const uint8_t* cur = blob.data();
        get(cur, pl.level_off, h.n_levels + 1);
        get(cur, pl.level_rare, h.n_levels);
        get(cur, pl.loads, h.n_loads);
        get(cur, p.asserts, h.n_asserts);
        get(cur, p.const_limbs, h.n_consts * h.nlimb);
        get(cur, p.const_unreduced, h.n_consts);
        get(cur, const_raw_flat, h.const_raw_bytes);
        get(cur, p.modulus_le, h.modulus_len);
        std::vector<char> pend;
        get(cur, pend, h.pending_len);
        get(cur, pl.group_descs, h.n_group_descs);
        get(cur, pl.group_ops, h.n_group_ops);
        get(cur, pl.group_tables, h.n_group_tables);
        get(cur, pl.depth_off, h.n_depth_off);
        get(cur, pl.group_hints, h.n_group_hints);
        get(cur, pl.hint_off, h.n_depth_off);
        pl.group_regs = (uint32_t)h.group_regs;
        pl.callout_slot0 = (uint32_t)h.callout_slot0;
        pl.n_callouts = (uint32_t)h.n_callouts;
        const uint8_t* q = const_raw_flat.data();
        p.const_raw.resize(h.n_consts);
        for (uint64_t i = 0; i < h.n_consts && q < const_raw_flat.data() + const_raw_flat.size(); i++) {
            uint32_t len;
            memcpy(&len, q, 4);
            p.const_raw[i].assign(q + 4, q + 4 + len);
            q += 4 + len;
        }
        p.field_set = true;
        p.modulus = BigU::from_bytes_le(p.modulus_le.data(), p.modulus_le.size());
        p.binary = h.binary != 0;
        p.nlimb = (int)h.nlimb;
        p.fp = h.fp;
        p.n_instance = h.n_instance;
        p.n_witness = h.n_witness;
        p.ir_gates = h.ir_gates;
        memcpy(p.cb_count, h.cb_count, sizeof h.cb_count);
        pl.n_slots = h.n_slots;
        pl.n_levels = (uint32_t)h.n_levels;
        pl.n_raw_ops = h.n_raw_ops;
        pl.algo_bytes_per_witness = h.algo_bytes_per_witness;
        pl.n_reused_slots = h.n_reused_slots;
        pl.max_level_ops = h.max_level_ops;
        memcpy(pl.n_dev_ops, h.n_dev_ops, sizeof h.n_dev_ops);
        c->is_boolean = h.is_boolean != 0;
        c->has_pending = h.has_pending != 0;
        c->pending_error.assign(pend.begin(), pend.end());
        c->keep_all = h.keep_all != 0;
        c->const_raw_stride = h.const_raw_stride;
        c->replica_n_ops = h.n_ops;
        c->replica_n_values = h.n_values;
        c->is_replica = true;
        c->finalized = true;
        c->inputs_uploaded = false;
        c->resident_tile = -1;
        c->flat_scope.clear();
        capture_reset(c, false);  // the device ops are about to be replaced
    }
    lap("unpack");
    // 3. the device plan, device to device; the root sends its ops as the plan made them, without its capture list's changes
    if (is_root) capture_mark_sinks(c, true);
    rc = bcast_array(c, c->d_ops, h.n_ops, root, is_root);
    if (is_root) capture_mark_sinks(c, false);
    if (rc != ZKB_OK) return rc;
    if ((rc = bcast_array(c, c->d_aseq, h.n_ops, root, is_root)) != ZKB_OK) return rc;
    if ((rc = bcast_array(c, c->d_loads, h.n_loads, root, is_root)) != ZKB_OK) return rc;
    if ((rc = bcast_array(c, c->d_consts, h.n_consts * h.nlimb, root, is_root)) != ZKB_OK) return rc;  // already in Montgomery form
    if ((rc = bcast_array(c, c->d_level_off, h.n_levels + 1, root, is_root)) != ZKB_OK) return rc;
    if ((rc = bcast_array(c, c->d_const_flags, h.has_const_flags ? h.n_consts : 0, root, is_root)) != ZKB_OK) return rc;
    if ((rc = bcast_array(c, c->d_const_raw, (size_t)h.const_raw_stride * h.n_consts, root, is_root)) != ZKB_OK) return rc;
    if (!is_root && (rc = ctx_upload_groups(c)) != ZKB_OK) return rc;  // small: from the host copy that came with the tables
    CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    lap("device plan");
    // the per-value tables (value -> slot / readable / kind / operand b) stay ON THE DEVICE of a replica: zkb_read_values
    // gathers the few entries a request names, so no peer pays a device-to-host copy of tables as long as the program
    {
        uint32_t *t_slot = c->d_tab_slot, *t_opb = c->d_tab_opb;
        uint8_t *t_read = c->d_tab_readable, *t_kind = c->d_tab_kind;
        const bool own = is_root && !c->is_replica;  // a recording root uploads its host tables for the duration of the broadcast
        if (own) {
            t_slot = t_opb = nullptr;
            t_read = t_kind = nullptr;
            const size_t n = h.n_values;
            if (n) {
                CUDA_TRY(c, cudaMalloc((void**)&t_slot, n * 4));
                CUDA_TRY(c, cudaMalloc((void**)&t_opb, n * 4));
                CUDA_TRY(c, cudaMalloc((void**)&t_read, n));
                CUDA_TRY(c, cudaMalloc((void**)&t_kind, n));
                CUDA_TRY(c, cudaMemcpyAsync(t_slot, pl.slot_of_value.data(), n * 4, cudaMemcpyHostToDevice, c->stream));
                CUDA_TRY(c, cudaMemcpyAsync(t_opb, p.opb.data(), n * 4, cudaMemcpyHostToDevice, c->stream));
                CUDA_TRY(c, cudaMemcpyAsync(t_read, pl.readable.data(), n, cudaMemcpyHostToDevice, c->stream));
                CUDA_TRY(c, cudaMemcpyAsync(t_kind, p.kind.data(), n, cudaMemcpyHostToDevice, c->stream));
            }
        }
        if ((rc = bcast_array(c, t_slot, h.n_values, root, is_root)) != ZKB_OK) return rc;
        if ((rc = bcast_array(c, t_opb, h.n_values, root, is_root)) != ZKB_OK) return rc;
        if ((rc = bcast_array(c, t_read, h.n_values, root, is_root)) != ZKB_OK) return rc;
        if ((rc = bcast_array(c, t_kind, h.n_values, root, is_root)) != ZKB_OK) return rc;
        CUDA_TRY(c, cudaStreamSynchronize(c->stream));
        if (own) {
            cudaFree(t_slot);
            cudaFree(t_opb);
            cudaFree(t_read);
            cudaFree(t_kind);
        } else {
            c->d_tab_slot = t_slot;
            c->d_tab_opb = t_opb;
            c->d_tab_readable = t_read;
            c->d_tab_kind = t_kind;
        }
    }
    lap("value tables");
    cm->program_generation++;
    return ZKB_OK;
}

}  // namespace zkb

// ---------------------------------------------------------------------------------------------- C ABI
extern "C" int zkb_comm_unique_id(zkb_comm_id* out) {
    if (!out) return ZKB_E_ARG;
    static_assert(sizeof(ncclUniqueId) <= sizeof(zkb_comm_id), "zkb_comm_id too small");
    NcclApi* api = nccl_api();
    if (!api->error.empty()) return ZKB_E_CUDA;
    ncclUniqueId id;
    if (api->GetUniqueId(&id) != ncclSuccess) return ZKB_E_CUDA;
    memset(out, 0, sizeof *out);
    memcpy(out->bytes, &id, sizeof id);
    return ZKB_OK;
}

extern "C" int zkb_comm_init_rank(zkb_ctx* c, const zkb_comm_id* id, int n_ranks, int rank) {
    if (!c || !id || n_ranks < 1 || rank < 0 || rank >= n_ranks) return c ? c->fail(ZKB_E_ARG, "zkb_comm_init_rank: bad rank / size") : ZKB_E_ARG;
    if (!c->has_gpu) return c->fail(ZKB_E_CUDA, "no CUDA device in this context (there is no CPU fallback)");
    if (c->comm) return c->fail(ZKB_E_ARG, "this context already belongs to a communicator");
    NcclApi* api = nccl_api();
    if (!api->error.empty()) return c->fail(ZKB_E_CUDA, api->error);
    CUDA_TRY(c, cudaSetDevice(c->device));
    ncclUniqueId nid;
    memcpy(&nid, id->bytes, sizeof nid);
    ncclComm_t comm = nullptr;
    NCCL_TRY(c, api, api->CommInitRank(&comm, n_ranks, nid, rank));
    c->comm = new CommState();
    c->comm->rank = rank;
    c->comm->size = n_ranks;
    c->comm->nccl = comm;
    // NCCL connects lazily: the first collective pays for the channels.  Pay here, where the communicator is made.
    return comm_warm_up(c);
}

extern "C" int zkb_comm_init(zkb_ctx** ctxs, int n) {
    if (!ctxs || n < 1) return ZKB_E_ARG;
    zkb_ctx* c0 = ctxs[0];
    bool shared_device = false;
    for (int i = 0; i < n; i++) {
        if (!ctxs[i]) return c0 ? c0->fail(ZKB_E_ARG, "zkb_comm_init: null context") : ZKB_E_ARG;
        if (!ctxs[i]->has_gpu) return c0->fail(ZKB_E_CUDA, "no CUDA device in a context of the communicator (there is no CPU fallback)");
        if (ctxs[i]->comm) return c0->fail(ZKB_E_ARG, "a context already belongs to a communicator");
        for (int j = 0; j < i; j++) {
            if (ctxs[j] == ctxs[i]) return c0->fail(ZKB_E_ARG, "zkb_comm_init: the same context twice");
            shared_device |= ctxs[j]->device == ctxs[i]->device;
        }
    }
    std::vector<ncclComm_t> comms(n, nullptr);
    std::shared_ptr<LocalGroup> local;
    if (shared_device || getenv("ZKB_COMM_LOCAL")) {
        local = std::make_shared<LocalGroup>();
        local->size = n;
        local->buf.assign(n, nullptr);
        for (int i = 0; i < n; i++) local->device.push_back(ctxs[i]->device);
    } else if (n > 1) {
        NcclApi* api = nccl_api();
        if (!api->error.empty()) return c0->fail(ZKB_E_CUDA, api->error);
        std::vector<int> devs;
        for (int i = 0; i < n; i++) devs.push_back(ctxs[i]->device);
        NCCL_TRY(c0, api, api->CommInitAll(comms.data(), n, devs.data()));
    }
    for (int i = 0; i < n; i++) {
        ctxs[i]->comm = new CommState();
        ctxs[i]->comm->rank = i;
        ctxs[i]->comm->size = n;
        ctxs[i]->comm->nccl = comms[i];
        ctxs[i]->comm->local = local;
    }
    if (comms[0]) {  // connect the channels now (one thread per rank: a collective blocks until every rank has joined it)
        std::vector<int> rcs(n, ZKB_OK);
        std::vector<std::thread> th;
        for (int i = 1; i < n; i++) th.emplace_back([&, i] { rcs[i] = comm_warm_up(ctxs[i]); });
        rcs[0] = comm_warm_up(ctxs[0]);
        for (auto& t : th) t.join();
        for (int i = 0; i < n; i++)
            if (rcs[i] != ZKB_OK) return i ? c0->fail(rcs[i], "rank " + std::to_string(i) + ": " + ctxs[i]->err) : rcs[i];
    }
    return ZKB_OK;
}

extern "C" int zkb_comm_info(zkb_ctx* c, int* rank, int* n_ranks, int* transport, int* nccl_version) {
    if (!c->comm) return c->fail(ZKB_E_ARG, "this context is not part of a communicator");
    if (rank) *rank = c->comm->rank;
    if (n_ranks) *n_ranks = c->comm->size;
    if (transport) *transport = c->comm->nccl ? 1 : (c->comm->local ? 2 : 0);
    if (nccl_version) {
        *nccl_version = 0;
        if (c->comm->nccl) nccl_api()->GetVersion(nccl_version);
    }
    return ZKB_OK;
}

extern "C" int zkb_comm_broadcast_program(zkb_ctx* c, int root) {
    if (!c->comm) return c->fail(ZKB_E_ARG, "this context is not part of a communicator (zkb_comm_init / zkb_comm_init_rank)");
    if (root < 0 || root >= c->comm->size) return c->fail(ZKB_E_ARG, "zkb_comm_broadcast_program: root out of range");
    if (c->comm->size == 1) return c->finalized ? ZKB_OK : c->fail(ZKB_E_ARG, "zkb_comm_broadcast_program: the root's program is not finalized");
    return broadcast_program(c, root);
}

extern "C" int zkb_comm_run(zkb_ctx* c, uint32_t first, uint32_t n_total, zkb_verdict* out) {
    if (!c->comm) return c->fail(ZKB_E_ARG, "this context is not part of a communicator (zkb_comm_init / zkb_comm_init_rank)");
    return ctx_run(c, out, first, n_total, true);
}

extern "C" int zkb_comm_evaluate(zkb_ctx* c, const uint8_t* inst, uint64_t inst_set_stride, const uint8_t* wit, uint64_t wit_set_stride,
                                 uint32_t value_stride, uint32_t n_local, uint32_t first, uint32_t n_total, zkb_verdict* out) {
    if (!c->comm) return c->fail(ZKB_E_ARG, "this context is not part of a communicator (zkb_comm_init / zkb_comm_init_rank)");
    int rc = zkb_upload_inputs(c, inst, inst_set_stride, wit, wit_set_stride, value_stride, n_local);
    if (rc != ZKB_OK) return rc;
    rc = ctx_run(c, out, first, n_total, true);
    if (rc != ZKB_OK) return rc;
    ctx_finish_e2e_timing(c);
    return ZKB_OK;
}

// One process, N devices: the caller's thread fans out to one host thread per context (a context is one host thread + one
// device); each evaluates its contiguous block of the batch, the verdicts are MIN-reduced, rank 0's copy goes to `out`.
static int sharded(zkb_ctx** ctxs, int n, const uint8_t* inst, uint64_t iss, const uint8_t* wit, uint64_t wss, uint32_t value_stride,
                   uint32_t n_batch, zkb_verdict* out, bool upload) {
    if (!ctxs || n < 1 || !ctxs[0]) return ZKB_E_ARG;
    zkb_ctx* c0 = ctxs[0];
    for (int i = 0; i < n; i++)
        if (!ctxs[i] || !ctxs[i]->comm || ctxs[i]->comm->size != n || ctxs[i]->comm->rank != i)
            return c0->fail(ZKB_E_ARG, "zkb_evaluate_sharded: pass the contexts in the order given to zkb_comm_init");
    if (!c0->finalized) return c0->fail(ZKB_E_ARG, "zkb_finalize must be called on the first context before evaluation");
    if (n_batch < (uint32_t)n) return c0->fail(ZKB_E_ARG, "zkb_evaluate_sharded: fewer witnesses than devices");
    // replicas that have not seen this program yet receive it now (once per finalized program)
    bool need_bcast = false;
    for (int i = 1; i < n; i++) need_bcast |= !ctxs[i]->finalized || ctxs[i]->comm->program_generation != c0->comm->program_generation;
    need_bcast |= n > 1 && c0->comm->program_generation == 0;
    std::vector<int> rcs(n, ZKB_OK);
    auto fan_out = [&](auto fn) {
        std::vector<std::thread> th;
        for (int i = 1; i < n; i++) th.emplace_back([&, i] { rcs[i] = fn(i); });
        rcs[0] = fn(0);
        for (auto& t : th) t.join();
        for (int i = 0; i < n; i++)
            if (rcs[i] != ZKB_OK) {
                if (i) c0->err = "rank " + std::to_string(i) + ": " + ctxs[i]->err;
                return rcs[i];
            }
        return (int)ZKB_OK;
    };
    int rc;
    if (need_bcast && (rc = fan_out([&](int i) { return zkb_comm_broadcast_program(ctxs[i], 0); })) != ZKB_OK) return rc;
    auto lo_of = [&](int i) { return (uint32_t)((uint64_t)n_batch * i / n); };
    if (upload) {
        // argument errors are found by every rank alike (same program, same strides) BEFORE the collective starts
        rc = fan_out([&](int i) {
            uint32_t lo = lo_of(i), hi = lo_of(i + 1);
            return zkb_upload_inputs(ctxs[i], inst ? inst + (uint64_t)lo * iss : nullptr, iss, wit ? wit + (uint64_t)lo * wss : nullptr, wss,
                                     value_stride, hi - lo);
        });
        if (rc != ZKB_OK) return rc;
    } else {
        for (int i = 0; i < n; i++)
            if (!ctxs[i]->inputs_uploaded || ctxs[i]->n_batch != lo_of(i + 1) - lo_of(i))
                return c0->fail(ZKB_E_ARG, "zkb_run_sharded: the resident inputs are not this batch (zkb_evaluate_sharded first)");
    }
    rc = fan_out([&](int i) {
        int r = ctx_run(ctxs[i], i == 0 ? out : nullptr, lo_of(i), n_batch, true);
        if (r == ZKB_OK && upload) ctx_finish_e2e_timing(ctxs[i]);
        return r;
    });
    return rc;
}

extern "C" int zkb_evaluate_sharded(zkb_ctx** ctxs, int n, const uint8_t* inst, uint64_t inst_set_stride, const uint8_t* wit,
                                    uint64_t wit_set_stride, uint32_t value_stride, uint32_t n_batch, zkb_verdict* out) {
    return sharded(ctxs, n, inst, inst_set_stride, wit, wit_set_stride, value_stride, n_batch, out, true);
}

extern "C" int zkb_run_sharded(zkb_ctx** ctxs, int n, uint32_t n_batch, zkb_verdict* out) {
    return sharded(ctxs, n, nullptr, 0, nullptr, 0, 0, n_batch, out, false);
}
