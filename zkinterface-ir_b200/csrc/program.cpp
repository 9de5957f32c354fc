#include "program.h"

#include <string.h>

#include <stdio.h>
#include <stdlib.h>

#include <algorithm>
#include <memory>
#include <atomic>
#include <iterator>
#include <chrono>
#include <thread>

namespace zkb {

bool Program::set_field(const uint8_t* mod_le, size_t len, uint32_t degree, std::string& err) {
    BigU m = BigU::from_bytes_le(mod_le, len);
    // PlaintextBackend::set_field, evaluator.rs:866-875 — same two errors, same order
    if (m.is_zero()) {
        err = "Modulus cannot be zero.";
        return false;
    }
    if (degree != 1) {
        err = "Field should be of degree 1";
        return false;
    }
    if (field_set) {
        if (!(m == modulus) && n_values() > 0) {
            err = "zkb: the field characteristic changed between relation messages (unsupported on device)";
            return false;
        }
        if (m == modulus) return true;
    }
    if (m.is_one()) {
        // SURVEY.md §8a trap 10: p = 1 makes the reference's `exp` recurse forever on a Switch
        err = "zkb: modulus 1 is not a field (the reference would not terminate on a Switch)";
        return false;
    }
    if (m.bits() > 32 * kMaxLimbs) {
        err = "zkb: field characteristic wider than 256 bits is not supported on device";
        return false;
    }
    bool is_two = (m.w.size() == 1 && m.w[0] == 2);
    if (!m.bit(0) && !is_two) {
        err = "zkb: even modulus other than 2 is not supported on device (Montgomery form needs an odd modulus)";
        return false;
    }
    modulus = m;
    modulus_le.assign(mod_le, mod_le + len);
    binary = is_two;
    size_t bits = m.bits();
    nlimb = bits <= 32 ? 1 : bits <= 64 ? 2 : bits <= 128 ? 4 : 8;
    memset(&fp, 0, sizeof(fp));
    fp.nlimb = (uint32_t)nlimb;
    m.to_limbs(fp.p, kMaxLimbs);
    if (!binary) {
        // n0inv = -p^{-1} mod 2^32 (Newton iteration on the odd low limb)
        uint32_t p0 = fp.p[0], inv = 1;
        for (int i = 0; i < 5; i++) inv *= 2 - p0 * inv;
        fp.n0inv = (uint32_t)(0u - inv);
        fp.mul_form = (nlimb == 8 && fp.p[0] == 1u && fp.p[1] == 0xFFFFFFFFu) ? kMulFormLow64 : kMulFormGeneric;
        BigU R;
        R.w.assign((size_t)nlimb + 1, 0);
        R.w[nlimb] = 1;
        BigU Rm = R.mod(m);
        BigU R2 = BigU::mulmod(Rm, Rm, m);
        Rm.to_limbs(fp.one, kMaxLimbs);
        R2.to_limbs(fp.r2, kMaxLimbs);
    } else {
        fp.one[0] = 1;
        fp.r2[0] = 1;
    }
    field_set = true;
    return true;
}

uint32_t Program::intern_const(const uint8_t* le, size_t n) {
    while (n > 0 && le[n - 1] == 0) n--;
    std::string key((const char*)le, n);
    auto it = const_index.find(key);
    if (it != const_index.end()) return it->second;
    uint32_t idx = n_consts();
    BigU v = BigU::from_bytes_le(le, n);
    bool unreduced = field_set && (v >= modulus);
    BigU r = unreduced ? v.mod(modulus) : v;
    size_t base = const_limbs.size();
    const_limbs.resize(base + (size_t)std::max(nlimb, 1), 0);
    r.to_limbs(&const_limbs[base], std::max(nlimb, 1));
    const_unreduced.push_back(unreduced ? 1 : 0);
    const_raw.emplace_back();
    if (unreduced) const_raw.back().assign(le, le + n);
    const_index.emplace(std::move(key), idx);
    return idx;
}

std::vector<uint8_t> Program::minus_one_le() const {
    BigU m = modulus;
    m.sub(BigU(1));
    std::vector<uint8_t> out((size_t)nlimb * 4, 0);
    for (size_t i = 0; i < out.size(); i++) out[i] = (uint8_t)(m.limb(i / 4) >> (8 * (i % 4)));
    while (out.size() > 1 && out.back() == 0) out.pop_back();
    return out;
}

// Slots released after one wavefront arrive as a few ASCENDING runs (one per wavefront that allocated them: a
// wavefront hands out slots in increasing order), so ordering them is a handful of linear merges, not a sort.
struct ReleaseList {
    std::vector<uint32_t> slots;
    std::vector<size_t> run_start;  // offsets where a new ascending run begins
    uint32_t last_writer = 0xFFFFFFFFu;
    void push(uint32_t slot, uint32_t writer) {
        if (writer != last_writer) {
            run_start.push_back(slots.size());
            last_writer = writer;
        }
        slots.push_back(slot);
    }
    void merge_runs() {
        while (run_start.size() > 1) {
            std::vector<size_t> next;
            for (size_t r = 0; r < run_start.size(); r += 2) {
                next.push_back(run_start[r]);
                if (r + 1 < run_start.size()) {
                    size_t end = r + 2 < run_start.size() ? run_start[r + 2] : slots.size();
                    std::inplace_merge(slots.begin() + run_start[r], slots.begin() + run_start[r + 1], slots.begin() + end);
                }
            }
            run_start.swap(next);
        }
    }
};

static inline uint32_t dev_op_of(uint8_t k) {
    switch (k) {
        case V_ADD: return D_ADD;
        case V_MUL: return D_MUL;
        case V_ADDC: return D_ADDC;
        case V_MULC: return D_MULC;
        case V_AND: return D_AND;
        case V_XOR: return D_XOR;
        case V_NOT: return D_NOT;
        default: return D_OPS;
    }
}

// The passes of Plan::build that walk values in sorted (i.e. random) order wait on DRAM latency, not on arithmetic:
// a few threads multiply the misses in flight.  Every parallel pass produces exactly what its sequential form does
// (positions, slots and release order are derived from prefix sums, not from arrival order).
unsigned plan_threads() {
    static int v = -1;
    if (v < 0) {
        const char* e = getenv("ZKB_PLAN_THREADS");
        unsigned hw = std::thread::hardware_concurrency();
        v = e ? atoi(e) : (int)std::min(8u, hw ? hw : 1u);
        if (v < 1) v = 1;
    }
    return (unsigned)v;
}

// fn(chunk index, begin, end) over [0, n) cut into T equal chunks
template <class F>
static void parallel_chunks(unsigned T, uint64_t n, F fn) {
    if (T < 2 || n == 0) {
        fn(0u, (uint64_t)0, n);
        return;
    }
    const uint64_t chunk = (n + T - 1) / T;
    std::vector<std::thread> pool;
    for (unsigned t = 1; t < T; t++) {
        uint64_t b = std::min(n, t * chunk), e = std::min(n, (t + 1) * chunk);
        pool.emplace_back([=, &fn]() { fn(t, b, e); });
    }
    fn(0u, (uint64_t)0, std::min(n, chunk));
    for (auto& th : pool) th.join();
}

static inline void atomic_max_u32(uint32_t* p, uint32_t val) {
    uint32_t cur = __atomic_load_n(p, __ATOMIC_RELAXED);
    while (cur < val && !__atomic_compare_exchange_n(p, &cur, val, true, __ATOMIC_RELAXED, __ATOMIC_RELAXED)) {
    }
}

void Plan::build(const Program& prog, bool keep_all, const std::vector<uint32_t>* live_values) {
    const bool timing = getenv("ZKB_TIMING") != nullptr;
    auto t_last = std::chrono::steady_clock::now();
    auto lap = [&](const char* what) {
        if (!timing) return;
        auto now = std::chrono::steady_clock::now();
        fprintf(stderr, "  plan %-28s %.3f s\n", what, std::chrono::duration<double>(now - t_last).count());
        t_last = now;
    };
    const uint32_t n = prog.n_values();
    const unsigned T = n >= (1u << 18) ? plan_threads() : 1;
    const uint8_t* kind = prog.kind.data();
    const uint32_t* opa = prog.opa.data();
    const uint32_t* opb = prog.opb.data();

    std::vector<uint32_t> level(n);
    std::vector<uint8_t> used(n, 0);  // consumed by another value
    uint32_t max_level = 0;
    constexpr uint32_t kAhead = 16;  // operands are random earlier values: start their loads a few iterations early
    // level(v) = 1 + max(level(operands)) over values in program order.  The chain is sequential in principle, but the
    // operands of a random circuit lie far back: chunks of 2^10 values (2^15: 0.93 s, 2^12: 0.38 s, 2^10: 0.19 s, 2^8: 0.26 s for C3 on 8 threads) are handed to the threads in order, a thread publishes
    // how far into its chunk it has got, and a reader only waits when its operand sits in a chunk that is still being worked on
    // (it never waits on a later chunk, and every claimed chunk is worked to its end: no deadlock).  A circuit whose operands
    // are all recent (a window of a few thousand wires) degenerates to one thread at a time — no slower than the plain loop.
    constexpr uint32_t kChunkLog2 = 10, kChunk = 1u << kChunkLog2;
    const uint32_t n_chunks = (uint32_t)(((uint64_t)n + kChunk - 1) >> kChunkLog2);
    std::unique_ptr<std::atomic<uint32_t>[]> progress(new std::atomic<uint32_t>[n_chunks ? n_chunks : 1]);
    for (uint32_t i = 0; i < n_chunks; i++) progress[i].store(0, std::memory_order_relaxed);
    std::atomic<uint32_t> next_chunk{0};
    const unsigned Tl = T;  // (T is 1 below 2^18 values)
    std::vector<uint32_t> thread_max(Tl, 0);
    uint32_t* lvl = level.data();
    uint8_t* usd = used.data();
    auto level_worker = [&](unsigned t) {
        uint32_t local_max = 0;
        for (;;) {
            const uint32_t c = next_chunk.fetch_add(1, std::memory_order_relaxed);
            if (c >= n_chunks) break;
            const uint32_t b = c << kChunkLog2, e = (uint32_t)std::min<uint64_t>(n, (uint64_t)b + kChunk);
            auto level_of = [&](uint32_t u) -> uint32_t {
                const uint32_t cu = u >> kChunkLog2;
                if (cu != c) {
                    const uint32_t need = u - (cu << kChunkLog2) + 1;
                    // (more threads than free cores: the chunk's owner may be descheduled, so a waiter that has spun a while
                    // gives its time slice away instead of burning it — 2.1 s instead of 0.012 s measured with 32 threads on 16 cores)
                    for (uint32_t spins = 0; progress[cu].load(std::memory_order_acquire) < need; spins++) {
                        if (spins < 256) __builtin_ia32_pause();
                        else std::this_thread::yield();
                    }
                }
                __atomic_store_n(&usd[u], (uint8_t)1, __ATOMIC_RELAXED);
                return lvl[u];
            };
            for (uint32_t v = b; v < e; v++) {
                if (v + kAhead < e) {
                    __builtin_prefetch(&lvl[opa[v + kAhead] < n ? opa[v + kAhead] : 0]);
                    __builtin_prefetch(&lvl[opb[v + kAhead] < n ? opb[v + kAhead] : 0]);
                }
                const uint8_t k = kind[v];
                uint32_t lv = 0;
                if (k > V_WITNESS) {
                    // a group output (implicit value, program.h) is ready before the first wavefront, like an input, and always stored
                    uint32_t la = is_callout(opa[v]) ? 0 : level_of(opa[v]);
                    const bool two = (k == V_ADD || k == V_MUL || k == V_AND || k == V_XOR);
                    if (two && !is_callout(opb[v])) la = std::max(la, level_of(opb[v]));
                    lv = la + 1;
                    if (lv > local_max) local_max = lv;
                }
                lvl[v] = lv;
                if (Tl > 1 && ((v - b) & 255) == 255) progress[c].store(v - b + 1, std::memory_order_release);
            }
            progress[c].store(e - b, std::memory_order_release);
        }
        thread_max[t] = local_max;
    };
    if (Tl > 1) {
        std::vector<std::thread> pool;
        for (unsigned t = 1; t < Tl; t++) pool.emplace_back(level_worker, t);
        level_worker(0);
        for (auto& th : pool) th.join();
    } else {
        level_worker(0);
    }
    for (unsigned t = 0; t < Tl; t++) max_level = std::max(max_level, thread_max[t]);
    // what a call group reads is consumed (stored); groups only read level-0 values, so nothing else changes
    // (the loops of a nest usually read the same progressions: each distinct one is walked once)
    struct Progression {
        uint32_t base, stride, n;
        bool operator==(const Progression& o) const { return base == o.base && stride == o.stride && n == o.n; }
    };
    struct ProgressionHash {
        size_t operator()(const Progression& p) const { return ((size_t)p.base * 0x9E3779B97F4A7C15ull) ^ ((size_t)p.stride << 32) ^ p.n; }
    };
    std::unordered_map<Progression, std::pair<uint32_t, uint32_t>, ProgressionHash> progressions;  // -> (slot stride | kTableStride, table offset)
    for (const CallGroup& cg : prog.groups) {
        for (uint32_t h : cg.seeds)
            if (!is_callout(h)) used[h] = 1;
        for (size_t k = 0; k < cg.in_base.size(); k++) {
            const uint32_t b = cg.in_base[k], st = cg.in_stride[k];
            if (is_callout(b) || (cg.carried() && cg.carry[k])) continue;
            if (!progressions.emplace(Progression{b, st, st ? cg.n_calls : 1}, std::make_pair(0u, 0u)).second) continue;
            if (st == 0) used[b] = 1;
            else for (uint32_t c = 0; c < cg.n_calls; c++) used[b + st * c] = 1;
        }
    }
    lap("levels");
    // earliest assert per value (a value that is non-zero fails at its first assert)
    std::vector<uint32_t> aseq(n, kNoSeq);
    callout_assert_seq.clear();
    callout_assert_value.clear();
    for (size_t s = 0; s < prog.asserts.size(); s++) {
        uint32_t v = prog.asserts[s].value;
        if (v == kGroupAssertValue) continue;  // inside a call group: tested by the group kernel
        if (is_callout(v)) {  // AssertZero directly on a group output: a standalone test in wavefront 1
            callout_assert_seq.push_back((uint32_t)s);
            callout_assert_value.push_back(v);
        } else if (aseq[v] == kNoSeq) {
            aseq[v] = (uint32_t)s;  // asserts are in program order: first wins
        }
    }
    std::vector<uint8_t> observable;
    if (!keep_all) {
        observable.assign(n, 0);
        if (live_values) {
            const uint32_t* lv = live_values->data();
            uint8_t* obs = observable.data();
            parallel_chunks(live_values->size() >= (1u << 18) ? T : 1, live_values->size(),
                            [&](unsigned, uint64_t b, uint64_t e) {
                                for (uint64_t i = b; i < e; i++)
                                    if (!is_callout(lv[i])) obs[lv[i]] = 1;
                            });
        }
    }

    // standalone asserts on level-0 values run in level 1
    input_assert_seq.clear();
    input_assert_value.clear();
    for (uint32_t v = 0; v < n; v++)
        if (aseq[v] != kNoSeq && kind[v] <= V_WITNESS) {
            input_assert_seq.push_back(aseq[v]);
            input_assert_value.push_back(v);
        }
    if (!(input_assert_seq.empty() && callout_assert_seq.empty()) && max_level < 1) max_level = 1;
    n_levels = max_level;

    lap("asserts/observable");
    // counting sort of device ops by (level, opcode); per-thread histograms over contiguous chunks of the value list give
    // every thread its own starting offsets, so the placement below is stable (same order as a sequential sort)
    const size_t n_keys = (size_t)n_levels * D_OPS;
    const unsigned Tsort = (T > 1 && n_keys * T <= n / 4) ? T : 1;
    std::vector<std::vector<uint64_t>> hist(Tsort, std::vector<uint64_t>(n_keys, 0));
    parallel_chunks(Tsort, n, [&](unsigned t, uint64_t b, uint64_t e) {
        uint64_t* h = hist[t].data();
        for (uint64_t v = b; v < e; v++)
            if (kind[v] > V_WITNESS) h[(size_t)(level[v] - 1) * D_OPS + dev_op_of(kind[v])]++;
    });
    std::vector<uint64_t> cnt(n_keys + 1, 0);
    for (unsigned t = 0; t < Tsort; t++)
        for (size_t k = 0; k < n_keys; k++) cnt[k + 1] += hist[t][k];
    if (n_levels > 0)  // (a program of inputs only has no wavefront and, by the rule above, no standalone assertion)
        cnt[(size_t)0 * D_OPS + D_ASSERT + 1] += input_assert_seq.size() + callout_assert_seq.size();
    for (size_t i = 0; i < n_keys; i++) cnt[i + 1] += cnt[i];
    const uint64_t n_ops = cnt[n_keys];
    level_off.assign((size_t)n_levels + 1, 0);
    for (uint32_t l = 0; l <= n_levels; l++) level_off[l] = cnt[(size_t)l * D_OPS];
    level_rare.assign((size_t)n_levels, 0);
    for (uint32_t l = 0; l < n_levels; l++) level_rare[l] = cnt[(size_t)l * D_OPS + D_AND];
    max_level_ops = 0;
    for (uint32_t l = 0; l < n_levels; l++)
        max_level_ops = (uint32_t)std::max<uint64_t>(max_level_ops, level_off[l + 1] - level_off[l]);

    lap("histogram");
    // last wavefront that reads each value (kForever: must stay readable after the run)
    constexpr uint32_t kForever = 0xFFFFFFFFu;
    const bool reuse = !keep_all && slot_reuse;
    std::vector<uint32_t> last_use;
    if (reuse) {
        last_use.assign(n, 0);
        uint32_t* lu = last_use.data();
        parallel_chunks(T, n, [&](unsigned, uint64_t b, uint64_t e) {  // a maximum: order of the updates is irrelevant
            for (uint64_t v = b; v < e; v++) {
                if (v + kAhead < e) {
                    __builtin_prefetch(&lu[opa[v + kAhead] < n ? opa[v + kAhead] : 0], 1);
                    __builtin_prefetch(&lu[opb[v + kAhead] < n ? opb[v + kAhead] : 0], 1);
                }
                uint8_t k = kind[v];
                if (k <= V_WITNESS) continue;
                if (!is_callout(opa[v])) atomic_max_u32(&lu[opa[v]], level[v]);
                if ((k == V_ADD || k == V_MUL || k == V_AND || k == V_XOR) && !is_callout(opb[v])) atomic_max_u32(&lu[opb[v]], level[v]);
            }
        });
        for (uint32_t v : input_assert_value)
            if (last_use[v] < 1) last_use[v] = 1;
        parallel_chunks(T, n, [&](unsigned, uint64_t b, uint64_t e) {
            for (uint64_t v = b; v < e; v++)
                if (observable[v]) lu[v] = kForever;
        });
    }
    // slots released once wavefront l has run (re-usable from wavefront l + 1 on: inside one launch a slot is
    // never both read and written)
    std::vector<ReleaseList> release_after(reuse ? (size_t)n_levels + 1 : 0);
    std::vector<uint32_t> free_slots;  // ascending from free_head on: the lowest free slot is handed out first
    std::vector<uint32_t> free_spare;
    size_t free_head = 0;
    constexpr uint32_t kInputWriter = 0xFFFFFFFEu;
    readable.assign(n, 0);

    lap("last use");
    // pass 1: place values (order index) and assign slots in placement order
    slot_of_value.assign(n, kNoSlot);
    loads.clear();
    uint32_t next_slot = 0;
    for (uint32_t v = 0; v < n; v++)
        if (kind[v] <= V_WITNESS) {
            slot_of_value[v] = next_slot;
            loads.push_back(InputLoad{next_slot, kind[v], opb[v], 0});
            readable[v] = 1;  // inputs are read back from the raw streams / constant pool
            if (reuse && last_use[v] != kForever) release_after[last_use[v]].push(next_slot, kInputWriter);
            next_slot++;
        }
    // group outputs follow the inputs (whose slots stay 0 .. n_loads - 1: the raw-value flags are indexed by them), in index
    // order; they are never released
    callout_slot0 = next_slot;
    n_callouts = prog.n_callouts;
    next_slot += prog.n_callouts;
    // slots must follow the sorted order, so ops are walked by position: value_at[position] = value
    std::vector<uint32_t> value_at(n_ops, kNoSlot);
    {
        // start[t][key] = first position of thread t's values with that key
        std::vector<uint64_t> run(cnt.begin(), cnt.end() - 1);
        for (unsigned t = 0; t < Tsort; t++)
            for (size_t k = 0; k < n_keys; k++) {
                uint64_t c = hist[t][k];
                hist[t][k] = run[k];
                run[k] += c;
            }
        uint32_t* va = value_at.data();
        parallel_chunks(Tsort, n, [&](unsigned t, uint64_t b, uint64_t e) {
            uint64_t* cur = hist[t].data();
            for (uint64_t v = b; v < e; v++)
                if (kind[v] > V_WITNESS) va[cur[(size_t)(level[v] - 1) * D_OPS + dev_op_of(kind[v])]++] = (uint32_t)v;
        });
    }
    lap("placement");
    // Inside each opcode group of a wavefront's hot range, gates that read the same wire run back to back: ordered by a key
    // operand (the one more gates of the wavefront read; a on a tie; a for AddConstant / MulConstant), then by value.  Today's
    // value order puts the readers of a wire hundreds of thousands of gates apart, by when its row has left L2; side by side,
    // the repeat reads hit L2 (DESIGN.md section 4).  Slots are still handed out in position order, so every level keeps
    // one ascending slot range.  ZKB_OPERAND_ORDER=0: value order.
    const char* eo = getenv("ZKB_OPERAND_ORDER");
    if ((!eo || atoi(eo) != 0) && n_levels + 1 < (1u << 24)) {
        // readers of a wire in the current wavefront: (wavefront + 1) << 8 | count (saturating at 255) in the no longer needed
        // level array, so no pass resets it between wavefronts
        uint32_t* rd = level.data();
        parallel_chunks(T, n, [&](unsigned, uint64_t b, uint64_t e) { memset(rd + b, 0, (e - b) * 4); });
        std::vector<uint32_t> key_at(n_ops);
        struct Group {
            uint64_t lo, hi;
        };
        std::vector<Group> groups;
        for (uint32_t l = 0; l < n_levels; l++) {
            const uint64_t lo = level_off[l], hi = level_rare[l];
            if (hi - lo < 2) continue;
            for (uint32_t op = D_ADD; op <= D_MULC; op++) {
                const uint64_t gl = cnt[(size_t)l * D_OPS + op], gh = cnt[(size_t)l * D_OPS + op + 1];
                if (gh - gl >= 2) groups.push_back(Group{gl, gh});
            }
            const uint32_t st = (l + 1) << 8;
            const unsigned Tl = (T > 1 && hi - lo >= (1u << 16)) ? T : 1;
            auto two_input = [&](uint32_t v) { return kind[v] == V_ADD || kind[v] == V_MUL; };
            parallel_chunks(Tl, hi - lo, [&](unsigned, uint64_t b, uint64_t e) {
                auto bump = [&](uint32_t u) {
                    if (is_callout(u)) return;
                    uint32_t cur = __atomic_load_n(&rd[u], __ATOMIC_RELAXED);
                    for (;;) {
                        const uint32_t next = cur < st ? st + 1 : (cur & 255) == 255 ? cur : cur + 1;
                        if (next == cur || __atomic_compare_exchange_n(&rd[u], &cur, next, true, __ATOMIC_RELAXED, __ATOMIC_RELAXED))
                            break;
                    }
                };
                for (uint64_t i = lo + b; i < lo + e; i++) {
                    if (i + kAhead < lo + e) {
                        const uint32_t w = value_at[i + kAhead];
                        if (!is_callout(opa[w])) __builtin_prefetch(&rd[opa[w]], 1);
                        if (two_input(w) && !is_callout(opb[w])) __builtin_prefetch(&rd[opb[w]], 1);
                    }
                    const uint32_t v = value_at[i];
                    bump(opa[v]);
                    if (two_input(v)) bump(opb[v]);
                }
            });
            parallel_chunks(Tl, hi - lo, [&](unsigned, uint64_t b, uint64_t e) {
                auto readers = [&](uint32_t u) { return is_callout(u) ? 0u : rd[u] & 255; };
                for (uint64_t i = lo + b; i < lo + e; i++) {
                    const uint32_t v = value_at[i];
                    key_at[i] = two_input(v) && readers(opb[v]) > readers(opa[v]) ? opb[v] : opa[v];
                }
            });
        }
        // stable sort by key (value order inside a group is ascending already): LSD radix, 11-bit digits, largest group first
        std::sort(groups.begin(), groups.end(), [](const Group& x, const Group& y) {
            return x.hi - x.lo != y.hi - y.lo ? x.hi - x.lo > y.hi - y.lo : x.lo < y.lo;
        });
        std::atomic<size_t> next_group{0};
        const unsigned Tg = (unsigned)std::min<size_t>(T, groups.size());
        parallel_chunks(Tg, Tg, [&](unsigned, uint64_t, uint64_t) {  // one chunk per thread, groups from a shared queue
            std::vector<uint32_t> tk, tv;
            for (size_t gi; (gi = next_group.fetch_add(1, std::memory_order_relaxed)) < groups.size();) {
                const uint64_t m = groups[gi].hi - groups[gi].lo;
                uint32_t* key = key_at.data() + groups[gi].lo;
                uint32_t* val = value_at.data() + groups[gi].lo;
                uint32_t kmin = 0xFFFFFFFFu, kmax = 0;
                for (uint64_t i = 0; i < m; i++) {
                    kmin = std::min(kmin, key[i]);
                    kmax = std::max(kmax, key[i]);
                }
                tk.resize(m);
                tv.resize(m);
                uint32_t *sk = key, *sv = val, *dk = tk.data(), *dv = tv.data();
                for (uint32_t shift = 0; shift < 32 && ((kmax - kmin) >> shift) != 0; shift += 11) {
                    uint64_t c[2049] = {0};
                    for (uint64_t i = 0; i < m; i++) c[(((sk[i] - kmin) >> shift) & 2047) + 1]++;
                    for (int d = 0; d < 2048; d++) c[d + 1] += c[d];
                    for (uint64_t i = 0; i < m; i++) {
                        const uint64_t j = c[((sk[i] - kmin) >> shift) & 2047]++;
                        dk[j] = sk[i];
                        dv[j] = sv[i];
                    }
                    std::swap(sk, dk);
                    std::swap(sv, dv);
                }
                if (sv != val) memcpy(val, sv, m * 4);
            }
        });
        lap("operand order");
    }
    ops.assign(n_ops, GateOp{0, 0, 0, 0});
    op_assert_seq.assign(n_ops, kNoSeq);
    for (int i = 0; i < D_OPS; i++) n_dev_ops[i] = 0;
    std::vector<uint32_t> meta_of(n_ops, 0);
    n_reused_slots = 0;
    n_raw_ops = 0;
    n_sink_ops = 0;
    double t_free = 0, t_dist = 0;
    for (uint32_t l = 0; l < n_levels; l++) {
        auto tf0 = std::chrono::steady_clock::now();
        if (reuse) {  // wavefront l+1 may overwrite everything whose last reader ran in wavefront <= l
            ReleaseList& rel = release_after[l];
            if (!rel.slots.empty()) {
                rel.merge_runs();
                if (free_head == free_slots.size()) {  // nothing left over: the released list is the free list
                    free_slots.swap(rel.slots);
                } else {
                    free_spare.clear();  // capacity is kept from wavefront to wavefront: no fresh pages to fault in
                    free_spare.reserve(rel.slots.size() + (free_slots.size() - free_head));
                    std::merge(free_slots.begin() + free_head, free_slots.end(), rel.slots.begin(), rel.slots.end(),
                               std::back_inserter(free_spare));
                    free_slots.swap(free_spare);
                }
                free_head = 0;
                ReleaseList().slots.swap(rel.slots);
            }
        }
        t_free += std::chrono::duration<double>(std::chrono::steady_clock::now() - tf0).count();
        // The k-th stored value of the wavefront takes the k-th free slot (ascending), then fresh slots: positions come
        // from a prefix sum over chunks of the wavefront, so the chunks can be processed by different threads.
        const uint64_t lo = level_off[l], hi = level_off[l + 1];
        const unsigned Tl = (T > 1 && hi - lo >= (1u << 16)) ? T : 1;
        std::vector<uint64_t> stored(Tl + 1, 0), sinks(Tl, 0);
        // pass A: the store decision and the flags of every op
        parallel_chunks(Tl, hi - lo, [&](unsigned t, uint64_t b, uint64_t e) {
            uint64_t cnt_store = 0, cnt_sink = 0;
            for (uint64_t i = lo + b; i < lo + e; i++) {
                if (i + kAhead < lo + e) {  // values arrive in sorted, i.e. random, order: start their loads early
                    uint32_t va = value_at[i + kAhead];
                    if (va != kNoSlot) {
                        __builtin_prefetch(&kind[va]);
                        __builtin_prefetch(&aseq[va]);
                        __builtin_prefetch(&used[va]);
                        if (!keep_all) __builtin_prefetch(&observable[va]);
                    }
                }
                uint32_t v = value_at[i];
                if (v == kNoSlot) continue;  // standalone assert position
                uint32_t meta = dev_op_of(kind[v]);
                bool has_assert = aseq[v] != kNoSeq;
                if (has_assert) meta |= F_ASSERT;
                // stored unless nothing will ever read it: a value only tested by its own fused assertion, or
                // (with slot re-use on) a dead value — it is still computed
                bool store = keep_all || used[v] || observable[v] || (!has_assert && !reuse);
                if (!store) {
                    meta |= F_NOSTORE;
                } else {
                    cnt_store++;
                    if (!used[v]) {
                        meta |= F_SINK;
                        cnt_sink++;
                    }
                }
                meta_of[i] = meta;
            }
            stored[t + 1] = cnt_store;
            sinks[t] = cnt_sink;
        });
        for (unsigned t = 0; t < Tl; t++) {
            stored[t + 1] += stored[t];
            n_sink_ops += sinks[t];
        }
        const uint64_t n_free = free_slots.size() - free_head, n_store = stored[Tl];
        // pass B: hand out the slots, collect what each stored value releases later
        std::vector<std::vector<std::pair<uint32_t, uint32_t>>> released(Tl);  // (wavefront after which it is free, slot)
        parallel_chunks(Tl, hi - lo, [&](unsigned t, uint64_t b, uint64_t e) {
            uint64_t k = stored[t];
            if (reuse) released[t].reserve(stored[t + 1] - stored[t]);
            for (uint64_t i = lo + b; i < lo + e; i++) {
                if (i + kAhead < lo + e) {
                    uint32_t va = value_at[i + kAhead];
                    if (va != kNoSlot) {
                        if (reuse) __builtin_prefetch(&last_use[va]);
                        if (!keep_all) __builtin_prefetch(&observable[va]);
                        __builtin_prefetch(&slot_of_value[va], 1);
                        __builtin_prefetch(&readable[va], 1);
                    }
                }
                uint32_t v = value_at[i];
                if (v == kNoSlot || (meta_of[i] & F_NOSTORE)) continue;
                const uint32_t slot = k < n_free ? free_slots[free_head + k] : next_slot + (uint32_t)(k - n_free);
                k++;
                slot_of_value[v] = slot;
                readable[v] = keep_all || observable[v];
                if (reuse && last_use[v] != kForever) released[t].push_back({std::max(last_use[v], l + 1), slot});
            }
        });
        const uint64_t n_reused = std::min(n_store, n_free);
        n_reused_slots += n_reused;
        free_head += n_reused;
        next_slot += (uint32_t)(n_store - n_reused);
        auto td0 = std::chrono::steady_clock::now();
        for (unsigned t = 0; t < Tl; t++)  // chunk order = ascending slots: one ascending run per target list
            for (const auto& rs : released[t]) release_after[rs.first].push(rs.second, l);
        t_dist += std::chrono::duration<double>(std::chrono::steady_clock::now() - td0).count();
    }
    if (timing) fprintf(stderr, "  plan   (free-list merges %.3f s, release distribution %.3f s)\n", t_free, t_dist);
    n_slots = next_slot;
    lap("slot assignment");
    // pass 2: emit ops with operand slots
    {
        const unsigned Te = (T > 1 && n_ops >= (1u << 16)) ? T : 1;
        std::vector<std::vector<uint64_t>> dev_cnt(Te, std::vector<uint64_t>(D_OPS + 1, 0));  // [D_OPS]: raw ops
        parallel_chunks(Te, n_ops, [&](unsigned t, uint64_t b, uint64_t e) {
            uint64_t* dc = dev_cnt[t].data();
            for (uint64_t i = b; i < e; i++) {
                if (i + 2 * kAhead < e) {  // two-stage prefetch: the value's record, then its operands' slots
                    uint32_t v2 = value_at[i + 2 * kAhead];
                    if (v2 != kNoSlot) {
                        __builtin_prefetch(&opa[v2]);
                        __builtin_prefetch(&opb[v2]);
                        __builtin_prefetch(&kind[v2]);
                        __builtin_prefetch(&aseq[v2]);
                        __builtin_prefetch(&slot_of_value[v2]);
                    }
                    uint32_t v1 = value_at[i + kAhead];
                    if (v1 != kNoSlot) {
                        if (opa[v1] < n) __builtin_prefetch(&slot_of_value[opa[v1]]);
                        if (opb[v1] < n) __builtin_prefetch(&slot_of_value[opb[v1]]);
                    }
                }
                uint32_t v = value_at[i];
                if (v == kNoSlot) continue;
                uint8_t k = kind[v];
                GateOp g;
                g.meta = meta_of[i];
                g.a = slot_of(opa[v]);
                bool two = (k == V_ADD || k == V_MUL || k == V_AND || k == V_XOR);
                g.b = two ? slot_of(opb[v]) : opb[v];
                g.out = slot_of_value[v];
                const bool a_in = !is_callout(opa[v]) && kind[opa[v]] <= V_WITNESS;
                if (k == V_NOT && a_in) {  // not(input): the reference tests the RAW integer
                    g.meta |= F_RAW;
                    dc[D_OPS]++;
                }
                // and / xor act on the integers the reference holds: an input operand >= p takes part unreduced
                // (evaluator.rs:924-930).  Mod 2 only the low bit matters, residues are exact there.
                if ((k == V_AND || k == V_XOR) && !prog.binary) {
                    const bool b_in = !is_callout(opb[v]) && kind[opb[v]] <= V_WITNESS;
                    if (a_in) g.meta |= F_RAW;
                    if (b_in) g.meta |= F_RAWB;
                    if (a_in || b_in) dc[D_OPS]++;
                }
                ops[i] = g;
                op_assert_seq[i] = aseq[v];
                dc[g.meta & 0xff]++;
            }
        });
        for (unsigned t = 0; t < Te; t++) {
            for (int k = 0; k < D_OPS; k++) n_dev_ops[k] += dev_cnt[t][k];
            n_raw_ops += dev_cnt[t][D_OPS];
        }
    }
    if (n_levels > 0) {
        uint64_t p = cnt[(size_t)0 * D_OPS + D_ASSERT];
        for (size_t i = 0; i < input_assert_seq.size(); i++, p++) {
            GateOp g;
            g.meta = D_ASSERT | F_ASSERT | F_NOSTORE | F_RAW;
            n_raw_ops++;
            g.a = slot_of_value[input_assert_value[i]];
            g.b = 0;
            g.out = kNoSlot;
            ops[p] = g;
            op_assert_seq[p] = input_assert_seq[i];
            n_dev_ops[D_ASSERT]++;
        }
        for (size_t i = 0; i < callout_assert_seq.size(); i++, p++) {  // a group output is a reduced value: no raw flag
            GateOp g;
            g.meta = D_ASSERT | F_ASSERT | F_NOSTORE;
            g.a = slot_of(callout_assert_value[i]);
            g.b = 0;
            g.out = kNoSlot;
            ops[p] = g;
            op_assert_seq[p] = callout_assert_seq[i];
            n_dev_ops[D_ASSERT]++;
        }
    }
    // call groups -> device descriptors, launch order = depth order (stable inside a depth)
    group_descs.clear();
    group_ops.clear();
    group_tables.clear();
    group_hints.clear();
    hint_off.clear();
    depth_off.clear();
    group_regs = 0;
    chain_descs.clear();
    chain_carry.clear();
    chain_off.clear();
    chain_regs = 0;
    if (!prog.groups.empty()) {
        std::vector<uint32_t> tmpl_off(prog.templates.size());
        for (size_t t = 0; t < prog.templates.size(); t++) {
            group_regs = std::max(group_regs, prog.templates[t].n_regs);
            tmpl_off[t] = (uint32_t)group_ops.size();
            uint32_t prev_dst = 0xFFFFFFFFu;
            const uint32_t n_asserts = (uint32_t)prog.templates[t].assert_wire.size();
            for (const TmplOp& o : prog.templates[t].ops) {
                GroupOp g{};
                if (!prog.binary) {  // register numbers and the op (program.h, GroupOp over a prime field)
                    const bool two = o.kind == V_ADD || o.kind == V_MUL;
                    switch (o.kind) {
                        case V_ADD: g.m_and = AG_ADD; break;
                        case V_MUL: g.m_and = AG_MUL; break;
                        case V_ADDC: g.m_and = AG_ADDC; g.m_xor = o.b; break;
                        case V_MULC: g.m_and = AG_MULC; g.m_xor = o.b; break;
                        case V_CONST: g.m_and = AG_CONST; g.m_xor = o.b; break;
                        default: g.m_and = AG_ASSERT; g.m_a = o.b; g.m_c = n_asserts; break;  // T_ASSERT
                    }
                    g.dst_off = o.kind == T_ASSERT ? 0 : o.dst;
                    g.a_off = o.kind == V_CONST ? 0 : o.a;
                    g.b_off = two ? o.b : g.a_off;
                    if (o.kind != V_CONST && prev_dst != 0xFFFFFFFFu) {
                        if (o.a == prev_dst) g.fwd |= 1;
                        if (two && o.b == prev_dst) g.fwd |= 2;
                    }
                    if (o.kind != T_ASSERT) prev_dst = o.dst;  // an assertion writes nothing: the held result stays
                    group_ops.push_back(g);
                    continue;
                }
                const uint32_t all = 0xFFFFFFFFu;
                const bool two = o.kind == V_ADD || o.kind == V_MUL || o.kind == V_AND || o.kind == V_XOR;
                const uint32_t cmask = (o.kind == V_CONST || o.kind == V_ADDC || o.kind == V_MULC)
                                           ? 0u - (prog.const_limbs[(size_t)o.b * prog.nlimb] & 1u) : 0u;
                g.dst_off = o.dst * kGroupThreads * 4;
                g.a_off = (o.kind == V_CONST ? o.dst : o.a) * kGroupThreads * 4;  // a constant reads nothing meaningful: masks are 0
                g.b_off = two ? o.b * kGroupThreads * 4 : g.a_off;
                switch (o.kind) {
                    case V_ADD: case V_XOR: g.m_xor = all; break;
                    case V_MUL: case V_AND: g.m_and = all; break;
                    case V_NOT: g.m_a = all; g.m_c = all; break;
                    case V_ADDC: g.m_a = all; g.m_c = cmask; break;
                    case V_MULC: g.m_a = cmask; break;
                    default: g.m_c = cmask; break;  // V_CONST
                }
                if (o.kind != V_CONST && prev_dst != 0xFFFFFFFFu) {
                    if (o.a == prev_dst) g.fwd |= 1;
                    if ((two ? o.b : o.a) == prev_dst) g.fwd |= 2;
                }
                prev_dst = o.dst;
                group_ops.push_back(g);
            }
        }
        uint32_t max_depth = 0;
        for (const CallGroup& cg : prog.groups) max_depth = std::max(max_depth, cg.depth);
        depth_off.assign((size_t)max_depth + 2, 0);
        chain_off.assign((size_t)max_depth + 2, 0);
        for (const CallGroup& cg : prog.groups) (cg.carried() ? chain_off : depth_off)[cg.depth + 1]++;
        for (size_t d = 0; d + 1 < depth_off.size(); d++) {
            depth_off[d + 1] += depth_off[d];
            chain_off[d + 1] += chain_off[d];
        }
        std::vector<uint32_t> cursor(depth_off.begin(), depth_off.end() - 1), calls_before((size_t)max_depth + 1, 0);
        std::vector<uint32_t> chain_cursor(chain_off.begin(), chain_off.end() - 1);
        group_descs.resize(depth_off.back());
        chain_descs.resize(chain_off.back());
        chain_carry.assign(chain_descs.size() * kMaxGroupInputs, 0);
        for (const CallGroup& cg : prog.groups) {
            const Template& tp = prog.templates[cg.tmpl];
            GroupDesc gd{};
            gd.tmpl_off = tmpl_off[cg.tmpl];
            gd.n_ops = (uint32_t)tp.ops.size();
            gd.n_out = tp.n_out;
            gd.n_in = tp.n_in;
            gd.n_calls = cg.n_calls;
            gd.out_slot = callout_slot0 + cg.first_callout;
            gd.pad = prog.binary ? 0 : cg.seq0;
            const uint32_t chain = cg.carried() ? chain_cursor[cg.depth]++ : 0;
            if (cg.carried()) {
                gd.first_call = tp.n_regs + cg.ring_regs;
                chain_regs = std::max(chain_regs, gd.first_call + tp.n_in * kChainStages);
            } else {
                gd.first_call = calls_before[cg.depth];
                calls_before[cg.depth] += cg.n_calls;
            }
            const uint32_t* seed = cg.seeds.data();
            for (uint32_t k = 0; k < tp.n_in; k++) {
                const uint32_t b = cg.in_base[k], st = cg.in_stride[k];
                if (cg.carried() && cg.carry[k]) {  // the seeds' slots, then the ring past the template's registers
                    const uint32_t w = cg.carry[k], lag = (w >> 8) & 0xFF;
                    gd.in_base[k] = (uint32_t)group_tables.size();
                    for (uint32_t s = 0; s < lag; s++) group_tables.push_back(slot_of(*seed++));
                    chain_carry[(size_t)chain * kMaxGroupInputs + k] = (w & ~(0x7FFFu << 16)) | ((tp.n_regs + ((w >> 16) & 0x7FFF)) << 16);
                    continue;
                }
                if (is_callout(b)) {  // outputs of earlier groups: consecutive indices are consecutive slots
                    gd.in_base[k] = slot_of(b);
                    gd.in_stride[k] = st;
                    continue;
                }
                const uint32_t s0 = slot_of_value[b];
                auto& memo = progressions[Progression{b, st, st ? cg.n_calls : 1}];  // (slot stride + 1 | 0: not looked at yet, table)
                if (memo.first == 0) {
                    bool affine = true;
                    uint32_t sst = 0;
                    if (cg.n_calls > 1 && st != 0) {
                        sst = slot_of_value[b + st] - s0;
                        for (uint32_t c = 2; c < cg.n_calls && affine; c++) affine = slot_of_value[b + st * c] == s0 + sst * c;
                    }
                    if (affine && sst < kTableStride - 1) {
                        memo.first = sst + 1;
                    } else {  // one table per distinct progression, shared by the groups that read it
                        memo.first = kTableStride;
                        memo.second = (uint32_t)group_tables.size();
                        for (uint32_t c = 0; c < cg.n_calls; c++) group_tables.push_back(slot_of_value[b + st * c]);
                    }
                }
                if (memo.first != kTableStride) {
                    gd.in_base[k] = s0;
                    gd.in_stride[k] = memo.first - 1;
                } else {
                    gd.in_base[k] = memo.second;
                    gd.in_stride[k] = kTableStride;
                }
            }
            if (cg.carried()) chain_descs[chain] = gd;
            else group_descs[cursor[cg.depth]++] = gd;
        }
        // thread -> group: a hint per 2^kGroupHintShift calls of a launch, then a short forward walk over first_call
        group_hints.clear();
        hint_off.assign(depth_off.size(), 0);
        for (size_t d = 0; d + 1 < depth_off.size(); d++) {
            hint_off[d] = (uint32_t)group_hints.size();
            const uint32_t lo = depth_off[d], hi = depth_off[d + 1];
            if (hi == lo) continue;
            const uint64_t calls = (uint64_t)group_descs[hi - 1].first_call + group_descs[hi - 1].n_calls;
            uint32_t g = 0;
            for (uint64_t c0 = 0; c0 < calls; c0 += (1u << kGroupHintShift)) {
                while (lo + g + 1 < hi && group_descs[lo + g + 1].first_call <= c0) g++;
                group_hints.push_back(g);
            }
        }
        hint_off[depth_off.size() - 1] = (uint32_t)group_hints.size();
    }
    lap("emit");
    const uint64_t E = prog.binary ? 1 : (uint64_t)prog.nlimb * 4;
    const uint64_t* c = prog.cb_count;
    algo_bytes_per_witness = 3 * E * (c[CB_ADD] + c[CB_MUL] + c[CB_AND] + c[CB_XOR]) +
                             2 * E * (c[CB_ADDC] + c[CB_MULC] + c[CB_NOT]) + E * c[CB_ASSERT_ZERO];
}

}  // namespace zkb
