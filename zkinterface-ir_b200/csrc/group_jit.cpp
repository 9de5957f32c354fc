// Run-time specialisation of the call-group kernel (program.h CallGroup; kernels.cu k_bool_groups is the interpreter).
//
// The interpreter keeps a call's registers in shared memory because a register FILE cannot be indexed dynamically: 2 LDS + 1
// STS per op and word make it LSU-bound (ncu: l1tex 92 % busy, C5 at 4096 witnesses 0.57 of the HBM copy peak).  The bodies are
// tiny and fixed once the relation is recorded, so the plan's templates are written out as straight-line CUDA — every op one
// expression over named variables, the masks of its GroupOp folded in as literals — and compiled for sm_100a with NVRTC on a
// background thread while the statement is already being evaluated by the interpreter; when the cubin is there the next
// pass loads it (driver API) and the groups run with their registers in REGISTERS: inputs in, bitwise ops, outputs out.
// Nothing here is needed for correctness: no NVRTC, a compile error or a failed load leave the interpreter in charge.
#include <dlfcn.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <map>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "context.h"

namespace zkb {

struct GroupJit {
    std::thread worker;
    std::atomic<int> state{0};  // 0 compiling, 2 cubin ready, 3 module loaded, -1 unavailable / failed
    std::vector<char> cubin;
    std::string log, source;
    void* module = nullptr;     // CUmodule
    void* fn[2] = {nullptr, nullptr};  // CUfunction: one word / four words per thread
    double compile_s = 0;
};

namespace {

struct Nvrtc {
    void* h = nullptr;
    int (*CreateProgram)(void**, const char*, const char*, int, const char* const*, const char* const*) = nullptr;
    int (*CompileProgram)(void*, int, const char* const*) = nullptr;
    int (*GetCUBINSize)(void*, size_t*) = nullptr;
    int (*GetCUBIN)(void*, char*) = nullptr;
    int (*GetProgramLogSize)(void*, size_t*) = nullptr;
    int (*GetProgramLog)(void*, char*) = nullptr;
    int (*DestroyProgram)(void**) = nullptr;
    bool ok = false;
};
Nvrtc* nvrtc() {
    static Nvrtc n;
    static std::atomic<bool> tried{false};
    static std::mutex* mu = new std::mutex();
    std::lock_guard<std::mutex> lk(*mu);
    if (tried) return &n;
    tried = true;
    const char* names[] = {getenv("ZKB_NVRTC_LIB"), "libnvrtc.so.12", "libnvrtc.so", "/usr/local/cuda/lib64/libnvrtc.so.12"};
    for (const char* nm : names) {
        if (!nm) continue;
        n.h = dlopen(nm, RTLD_NOW | RTLD_LOCAL);
        if (n.h) break;
    }
    if (!n.h) return &n;
#define BIND(field, sym) *(void**)(&n.field) = dlsym(n.h, sym)
    BIND(CreateProgram, "nvrtcCreateProgram");
    BIND(CompileProgram, "nvrtcCompileProgram");
    BIND(GetCUBINSize, "nvrtcGetCUBINSize");
    BIND(GetCUBIN, "nvrtcGetCUBIN");
    BIND(GetProgramLogSize, "nvrtcGetProgramLogSize");
    BIND(GetProgramLog, "nvrtcGetProgramLog");
    BIND(DestroyProgram, "nvrtcDestroyProgram");
#undef BIND
    n.ok = n.CreateProgram && n.CompileProgram && n.GetCUBINSize && n.GetCUBIN && n.GetProgramLogSize && n.GetProgramLog && n.DestroyProgram;
    return &n;
}

struct Driver {
    void* h = nullptr;
    int (*ModuleLoadData)(void**, const void*) = nullptr;
    int (*ModuleGetFunction)(void**, void*, const char*) = nullptr;
    int (*ModuleUnload)(void*) = nullptr;
    int (*LaunchKernel)(void*, unsigned, unsigned, unsigned, unsigned, unsigned, unsigned, unsigned, void*, void**, void**) = nullptr;
    bool ok = false;
};
Driver* driver() {
    static Driver d;
    static std::atomic<bool> tried{false};
    static std::mutex* mu = new std::mutex();
    std::lock_guard<std::mutex> lk(*mu);
    if (tried) return &d;
    tried = true;
    d.h = dlopen("libcuda.so.1", RTLD_NOW | RTLD_LOCAL);
    if (!d.h) return &d;
    *(void**)(&d.ModuleLoadData) = dlsym(d.h, "cuModuleLoadData");
    *(void**)(&d.ModuleGetFunction) = dlsym(d.h, "cuModuleGetFunction");
    *(void**)(&d.ModuleUnload) = dlsym(d.h, "cuModuleUnload");
    *(void**)(&d.LaunchKernel) = dlsym(d.h, "cuLaunchKernel");
    d.ok = d.ModuleLoadData && d.ModuleGetFunction && d.ModuleUnload && d.LaunchKernel;
    return &d;
}

// one template = one `case` of the kernel's switch on GroupDesc::tmpl_off
struct TemplateShape {
    uint32_t n_ops, n_out, n_in;
};

std::string hex(uint32_t v) {
    char b[16];
    snprintf(b, sizeof b, "0x%08xu", v);
    return b;
}

// the op as an expression over named registers, masks folded: r = (a & b & m_and) ^ ((a ^ b) & m_xor) ^ (a & m_a) ^ m_c
std::string op_expr(const GroupOp& g) {
    const std::string a = "r" + std::to_string(g.a_off / (kGroupThreads * 4)), b = "r" + std::to_string(g.b_off / (kGroupThreads * 4));
    std::vector<std::string> terms;
    auto masked = [](const std::string& e, uint32_t m) { return m == 0xFFFFFFFFu ? e : "(" + e + " & S(" + hex(m) + "))"; };
    if (g.m_and) terms.push_back(masked("(" + a + " & " + b + ")", g.m_and));
    if (g.m_xor) terms.push_back(masked("(" + a + " ^ " + b + ")", g.m_xor));
    if (g.m_a) terms.push_back(masked(a, g.m_a));
    if (g.m_c) terms.push_back("S(" + hex(g.m_c) + ")");
    if (terms.empty()) return "S(0u)";
    std::string e = terms[0];
    for (size_t i = 1; i < terms.size(); i++) e += " ^ " + terms[i];
    return e;
}

std::string generate(const Plan& pl) {
    std::map<uint32_t, TemplateShape> shapes;
    for (const GroupDesc& d : pl.group_descs) shapes[d.tmpl_off] = TemplateShape{d.n_ops, d.n_out, d.n_in};
    std::string s;
    s += "typedef unsigned int u32;\ntypedef unsigned long long u64;\n";
    s += "struct GroupDesc { u32 tmpl_off, n_ops, n_out, n_in, n_calls, out_slot, first_call, pad; u32 in_base[8]; u32 in_stride[8]; };\n";
    s += "__device__ __forceinline__ uint4 operator^(uint4 a, uint4 b) { return make_uint4(a.x ^ b.x, a.y ^ b.y, a.z ^ b.z, a.w ^ b.w); }\n";
    s += "__device__ __forceinline__ uint4 operator&(uint4 a, uint4 b) { return make_uint4(a.x & b.x, a.y & b.y, a.z & b.z, a.w & b.w); }\n";
    s += "template <class V> struct Splat;\n";
    s += "template <> struct Splat<u32> { static __device__ __forceinline__ u32 of(u32 m) { return m; } };\n";
    s += "template <> struct Splat<uint4> { static __device__ __forceinline__ uint4 of(u32 m) { return make_uint4(m, m, m, m); } };\n";
    s += "#define S(m) Splat<V>::of(m)\n";
    s += "template <class V, int LOG2W>\n__device__ __forceinline__ void run(const GroupDesc* __restrict__ descs, u32 n_groups, u64 total_calls,\n"
         "        const u32* __restrict__ tables, const u32* __restrict__ hints, u32* __restrict__ store, u32 log2_words) {\n";
    s += "    const u32 log2_vecs = log2_words - LOG2W;\n    const u64 total = total_calls << log2_vecs;\n    const u32 vmask = (1u << log2_vecs) - 1;\n";
    s += "    V* vstore = reinterpret_cast<V*>(store);\n";
    s += "    for (u64 tid = blockIdx.x * (u64)blockDim.x + threadIdx.x; tid < total; tid += (u64)gridDim.x * blockDim.x) {\n";
    s += "        const u32 call_g = (u32)(tid >> log2_vecs), vw = (u32)tid & vmask;\n";
    s += "        u32 gi = __ldg(hints + (call_g >> " + std::to_string(kGroupHintShift) + "));\n";
    s += "        while (gi + 1 < n_groups && call_g >= __ldg(&descs[gi + 1].first_call)) gi++;\n";
    s += "        const GroupDesc* d = descs + gi;\n";
    s += "        const uint4 h0 = __ldg(reinterpret_cast<const uint4*>(d));\n        const uint4 h1 = __ldg(reinterpret_cast<const uint4*>(d) + 1);\n";
    s += "        const u32 call = call_g - h1.z;\n        const u64 out0 = (u64)h1.y + (u64)call * h0.z;\n";
    s += "        switch (h0.x) {\n";
    for (const auto& kv : shapes) {
        const uint32_t off = kv.first;
        const TemplateShape& t = kv.second;
        s += "        case " + std::to_string(off) + "u: {\n";
        // registers: every one the template names
        uint32_t n_regs = t.n_out + t.n_in;
        for (uint32_t i = 0; i < t.n_ops; i++) {
            const GroupOp& g = pl.group_ops[off + i];
            n_regs = std::max(n_regs, std::max(g.dst_off, std::max(g.a_off, g.b_off)) / (kGroupThreads * 4) + 1);
        }
        s += "            V";
        for (uint32_t r = 0; r < n_regs; r++) s += std::string(r ? ", " : " ") + "r" + std::to_string(r) + " = S(0u)";
        s += ";\n";
        for (uint32_t k0 = 0; k0 < t.n_in; k0 += 4) {
            const std::string q = std::to_string(k0 / 4);
            s += "            const uint4 b" + q + " = __ldg(reinterpret_cast<const uint4*>(d->in_base + " + std::to_string(k0) + "));\n";
            s += "            const uint4 s" + q + " = __ldg(reinterpret_cast<const uint4*>(d->in_stride + " + std::to_string(k0) + "));\n";
        }
        const char* comp[4] = {"x", "y", "z", "w"};
        for (uint32_t k = 0; k < t.n_in; k++) {
            const std::string q = std::to_string(k / 4), cpn = comp[k % 4];
            s += "            { const u32 bs = b" + q + "." + cpn + ", st = s" + q + "." + cpn + ";\n";
            s += "              const u32 slot = st == 0xFFFFFFFFu ? __ldg(tables + bs + call) : bs + st * call;\n";
            s += "              r" + std::to_string(t.n_out + k) + " = vstore[((u64)slot << log2_vecs) + vw]; }\n";
        }
        for (uint32_t i = 0; i < t.n_ops; i++) {
            const GroupOp& g = pl.group_ops[off + i];
            s += "            r" + std::to_string(g.dst_off / (kGroupThreads * 4)) + " = " + op_expr(g) + ";\n";
        }
        for (uint32_t k = 0; k < t.n_out; k++) s += "            vstore[((out0 + " + std::to_string(k) + ") << log2_vecs) + vw] = r" + std::to_string(k) + ";\n";
        s += "        } break;\n";
    }
    s += "        default: break;\n        }\n    }\n}\n";
    s += "extern \"C\" __global__ void __launch_bounds__(256) zkb_groups_w1(const GroupDesc* descs, u32 n_groups, u64 total_calls, const u32* tables,\n"
         "        const u32* hints, u32* store, u32 log2_words) { run<u32, 0>(descs, n_groups, total_calls, tables, hints, store, log2_words); }\n";
    s += "extern \"C\" __global__ void __launch_bounds__(256) zkb_groups_w4(const GroupDesc* descs, u32 n_groups, u64 total_calls, const u32* tables,\n"
         "        const u32* hints, u32* store, u32 log2_words) { run<uint4, 2>(descs, n_groups, total_calls, tables, hints, store, log2_words); }\n";
    return s;
}

void compile(GroupJit* j) {
    const auto t0 = std::chrono::steady_clock::now();
    Nvrtc* n = nvrtc();
    if (!n->ok) {
        j->log = "NVRTC is not available";
        j->state = -1;
        return;
    }
    void* prog = nullptr;
    if (n->CreateProgram(&prog, j->source.c_str(), "zkb_groups.cu", 0, nullptr, nullptr) != 0) {
        j->log = "nvrtcCreateProgram failed";
        j->state = -1;
        return;
    }
    const char* opts[] = {"--gpu-architecture=sm_100a", "--std=c++17"};
    const int rc = n->CompileProgram(prog, 2, opts);
    size_t ls = 0;
    if (n->GetProgramLogSize(prog, &ls) == 0 && ls > 1) {
        j->log.resize(ls);
        n->GetProgramLog(prog, &j->log[0]);
    }
    size_t cs = 0;
    if (rc != 0 || n->GetCUBINSize(prog, &cs) != 0 || cs == 0) {
        n->DestroyProgram(&prog);
        j->state = -1;
        return;
    }
    j->cubin.resize(cs);
    const int rg = n->GetCUBIN(prog, j->cubin.data());
    n->DestroyProgram(&prog);
    j->compile_s = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
    j->state = rg == 0 ? 2 : -1;
}

}  // namespace

// called when a plan with call groups has been uploaded: start the compilation (once per plan)
void group_jit_start(zkb_ctx* c) {
    group_jit_free(c);
    const char* e = getenv("ZKB_GROUP_JIT");
    const bool sync = e && atoi(e) == 2;  // compile in the calling thread (tests; also without a device: NVRTC needs none)
    if (c->plan.group_descs.empty()) return;
    if (!c->prog.binary) {  // prime-field templates are left to the interpreter kernel (k_arith_groups): state -1
        c->gjit = new GroupJit();
        c->gjit->state = -1;
        c->gjit->log = "call groups over a prime field run in the interpreter kernel";
        return;
    }
    if ((e && atoi(e) == 0) || (!c->has_gpu && !sync)) return;
    GroupJit* j = new GroupJit();
    c->gjit = j;
    j->source = generate(c->plan);
    if (sync) {
        compile(j);
        return;
    }
    j->worker = std::thread(compile, j);
}

void group_jit_free(zkb_ctx* c) {
    GroupJit* j = c->gjit;
    if (!j) return;
    if (j->worker.joinable()) j->worker.join();
    if (j->module && driver()->ok) driver()->ModuleUnload(j->module);
    delete j;
    c->gjit = nullptr;
}

// 0 compiling, 2 ready (loaded on the next pass), 3 loaded, -1 failed / unavailable, -2 no groups or switched off
int group_jit_wait(zkb_ctx* c) {
    GroupJit* j = c->gjit;
    if (!j) return -2;
    if (j->worker.joinable()) j->worker.join();
    return j->state;
}
int group_jit_state(zkb_ctx* c) { return c->gjit ? (int)c->gjit->state : -2; }
const char* group_jit_log(zkb_ctx* c) { return c->gjit ? c->gjit->log.c_str() : ""; }
const char* group_jit_source(zkb_ctx* c) { return c->gjit ? c->gjit->source.c_str() : ""; }
double group_jit_compile_seconds(zkb_ctx* c) { return c->gjit ? c->gjit->compile_s : 0; }

// launches the specialised kernel for one depth; false: not available (yet) — the caller runs the interpreter
bool group_jit_launch(zkb_ctx* c, const GroupDesc* d_descs, uint32_t n_groups, uint64_t total_calls, const uint32_t* d_hints, uint32_t log2_words,
                      void* stream) {
    GroupJit* j = c->gjit;
    if (!j || j->state < 2) return false;
    Driver* dr = driver();
    if (!dr->ok) {
        j->state = -1;
        return false;
    }
    if (j->state == 2) {  // first use: load the module into the current (primary) context
        if (j->worker.joinable()) j->worker.join();
        if (dr->ModuleLoadData(&j->module, j->cubin.data()) != 0 || dr->ModuleGetFunction(&j->fn[0], j->module, "zkb_groups_w1") != 0 ||
            dr->ModuleGetFunction(&j->fn[1], j->module, "zkb_groups_w4") != 0) {
            j->log += "\ncuModuleLoadData / cuModuleGetFunction failed";
            j->state = -1;
            return false;
        }
        j->state = 3;
    }
    const bool wide = log2_words >= 2;
    const uint64_t total = total_calls << (wide ? log2_words - 2 : log2_words);
    const uint64_t tiles = (total + 255) / 256;
    const unsigned grid = (unsigned)std::min<uint64_t>(tiles, (uint64_t)c->sm_count * 64);
    const uint32_t* tables = c->d_group_tables;
    void* args[] = {(void*)&d_descs, (void*)&n_groups, (void*)&total_calls, (void*)&tables, (void*)&d_hints, (void*)&c->d_store, (void*)&log2_words};
    return dr->LaunchKernel(j->fn[wide ? 1 : 0], grid, 1, 1, 256, 1, 1, 0, stream, args, nullptr) == 0;
}

}  // namespace zkb
